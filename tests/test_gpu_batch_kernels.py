"""Batched forward / log-probability on the decomposition shapes no other test sends through them: the two-stage DMMA
evaluator with 1-3 k chunks (<= 48 taus) and the FP64 column split over a 4-CTA cluster (512 taus, 64 frequencies).
Per-spectrum frequency and tau grids, 300 rows per spectrum (the last 128-row chunk ragged), enough spectra that every
CTA strides over several chunks, and 10 % of the rows outside the prior box; checked against the C oracle to 1e-12."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = [  # N, n_tau, spectra
    (64, 16, 400),
    (33, 32, 400),
    (20, 48, 400),
    (64, 512, 40),
]


@pytest.mark.parametrize("N,S,B", SHAPES, ids=[f"N{s[0]}-S{s[1]}" for s in SHAPES])
def test_batch_forward_logprob_match_oracle(N, S, B):
    from bisip_b200 import engine
    from bisip_b200.batch import BatchInversion, tau_grid
    from oracle import oracle
    rng = np.random.default_rng(S)
    n, pd = 300, 4
    w = np.stack([2 * np.pi * np.logspace(3.5, -1.5, N) * (1.0 + 0.01 * b) for b in range(B)])
    y = rng.normal(0.5, 0.2, (B, 2, N))
    yerr = rng.uniform(0.01, 0.05, (B, 2, N))
    inv = BatchInversion('decomp', w, y, yerr, nwalkers=16, nsteps=1, poly_deg=pd, n_tau=S)
    lo, hi = inv.param_bounds
    th = lo + (hi - lo) * rng.uniform(0.02, 0.98, (B, n, inv.ndim))
    th[:, :, 1:] *= 1.0 / 3.0 ** np.arange(inv.ndim - 1)
    out = np.nonzero(rng.random((B, n)) < 0.1)
    th[out[0], out[1], rng.integers(0, inv.ndim, len(out[0]))] = 2.0       # above every upper bound
    dev_th, dev_w = inv._to_dev(th, 0, B), inv._to_dev(w, 0, B)
    Z = engine.forward(inv._spec(), dev_th, dev_w).cpu().numpy()
    lp = engine.log_probability(inv._spec(), dev_th, dev_w, inv._to_dev(y, 0, B), inv._to_dev(yerr, 0, B),
                                inv._to_dev(inv.param_bounds[None], 0, 1)[0]).cpu().numpy()
    for b in (0, B // 2, B - 1):
        _, taus, log_taus = tau_grid(w[b], S, pd)
        prob = oracle.Problem('decomp', w[b], y[b], yerr[b], inv.param_bounds, taus=taus, log_taus=log_taus)
        Zo = prob.forward(th[b])
        assert (np.max(np.abs(Z[b] - Zo), axis=(1, 2)) / np.max(np.abs(Zo), axis=(1, 2))).max() <= 1e-12
        lpo = prob.log_probability(th[b])
        fin = np.isfinite(lpo)
        assert 0 < (~fin).sum() < n and np.array_equal(fin, np.isfinite(lp[b]))
        assert np.max(np.abs(lp[b][fin] - lpo[fin]) / np.maximum(1, np.abs(lpo[fin]))) <= 1e-12
