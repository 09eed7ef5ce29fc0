"""The exact fallback of the vector-model evaluators.

``vec_row_chi`` (bisip_b200/csrc/models.cuh) evaluates a row with ``rcp_fast`` and ``exp_fast``; when any element
leaves their range (``rcp_in_range``: den with biased exponent in [32, 2014], i.e. [2^-991, 2^992); ``|x| < 700`` for
the exponential), the whole row is evaluated again with true divisions and ``exp``.  The sampler kernels (both
families) and the batched log-probability go through this path.  Uniform starts inside the box never leave the
range, but these points inside the box do, and the reference is finite at all of them:

* Dias ``delta = 1e-150``: some elements in range, some finite out of range, some overflow to inf (a mixed row);
* Dias ``delta = 1e-300``: every element inf (the ``isinf(den)`` branch);
* Shin ``R1 = 1e-150``: finite but out of range;
* Shin ``R1 = 1e-300`` and ``R1 = 5e-324``: inf; at the second 1/R1 is inf itself and the kernel's 2^600 stand-in
  takes its place.

``m`` stays at 0.5: near 1, ``R0 - R0 m`` against ``R0 (1 - m)`` loses digits to cancellation.  Cole-Cole is left
out: inside its box ``|c (ln w + log_tau)| <= ~17`` and den >= 1, so its fallback cannot be reached.
"""
import numpy as np
import pytest

from helpers import lp_err, normwise, oracle_problem

pytestmark = pytest.mark.gpu

DIAS_PTS = np.array([[1.0, 0.5, -5.0, 10.0, 1e-150],
                     [1.0, 0.5, -5.0, 10.0, 1e-300]])
SHIN_PTS = np.array([[1e-150, 0.5, -14.0, -6.0, 0.5, 0.5],
                     [1e-300, 0.5, -14.0, -6.0, 0.5, 0.5],
                     [5e-324, 0.5, -14.0, -6.0, 0.5, 0.5]])
PTS = {'dias': DIAS_PTS, 'shin': SHIN_PTS}


def _in_range(den):
    with np.errstate(invalid='ignore'):
        return np.isfinite(den) & (den >= 2.0 ** -991) & (den < 2.0 ** 992)


def _den(model, th, w):
    """den of every element of the kernel's row (models.cuh DiasRow / ShinRow), restated in NumPy: (elements, N)."""
    with np.errstate(over='ignore', divide='ignore', invalid='ignore'):
        if model == 'dias':
            R0, m, log_tau, eta, delta = th
            tau = np.exp(log_tau)
            tau_p = tau * (1.0 / delta - 1.0) / (1.0 - m)
            sq = np.sqrt(w) * (tau * abs(eta) * 0.70710678118654752440)
            mre, mim = sq, w * tau + sq
            d = mre * mre + mim * mim
            wtp = w * tau_p
            ere, eim = wtp * mim, wtp * (d + mre)
            bre = d + ere
            return (bre * bre + eim * eim)[None]
        out = []
        for i in range(2):
            ir = 1.0 / th[i]
            ir = np.copysign(2.0 ** 600, ir) if np.isinf(ir) else ir
            x = np.exp(th[4 + i] * np.log(w))
            q = np.exp(th[2 + i])
            dre, dim = x * (q * np.cos(0.5 * np.pi * th[4 + i])) + ir, x * (q * np.sin(0.5 * np.pi * th[4 + i]))
            out.append(dre * dre + dim * dim)
        return np.array(out)


def _leaves_range(model, th, w):
    den = _den(model, th, w)
    return not np.all(_in_range(den))


@pytest.mark.parametrize("model", ['dias', 'shin'])
def test_fallback_points_forward_and_logprob_match_oracle(model, gold_fl, gold_ld, data_files):
    from helpers import make_model
    m = make_model(model, data_files['SIP-K389175'])
    prob = oracle_problem(model, gold_fl, gold_ld)
    w = m.data['w']
    pts = PTS[model]
    np.testing.assert_array_equal(m.param_bounds, prob.bounds)
    assert np.all((m.param_bounds[0] < pts) & (pts < m.param_bounds[1]))
    den = [_den(model, t, w) for t in pts]
    if model == 'dias':
        d0, d1 = den[0][0], den[1][0]
        assert _in_range(d0).any() and np.isinf(d0).any() and (np.isfinite(d0) & ~_in_range(d0)).any()   # mixed row
        assert np.isinf(d1).all()
    else:
        assert np.all(np.isfinite(den[0][0]) & ~_in_range(den[0][0]))
        assert np.isinf(den[1][0]).all() and np.isinf(den[2][0]).all()
        with np.errstate(over='ignore'):
            assert np.isinf(1.0 / pts[2, 0])
    Zo = prob.forward(pts)
    lpo = prob.log_probability(pts)
    assert np.all(np.isfinite(Zo)) and np.all(np.isfinite(lpo))
    assert normwise(m.forward(pts, w), Zo).max() <= 1e-12
    args = (m.data['w'], m.data['zn'], m.data['zn_err'])
    assert lp_err(m._log_probability(pts, m.forward, m.param_bounds, *args), lpo).max() <= 1e-12
    assert lp_err(m._log_likelihood(pts, m.forward, *args), lpo).max() <= 1e-12


SAMPLER_CASES = [  # model, data, walkers, steps: warp-private (W <= 64) and block-synchronous (W > 64, N > 32) kernels
    ('dias', 'file', 32, 20),
    ('dias', 'syn', 96, 10),
    ('shin', 'file', 32, 20),
    ('shin', 'syn', 96, 10),
]


@pytest.mark.parametrize("model,data,W,T", SAMPLER_CASES, ids=[f"{c[0]}-{c[1]}-W{c[2]}" for c in SAMPLER_CASES])
def test_fallback_points_in_sampler_match_oracle(model, data, W, T, gold_fl, gold_ld):
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    from oracle import oracle
    if data == 'file':
        w, zn, ze = (gold_ld[f'SIP-K389175/{k}'] for k in ('w', 'zn', 'zn_err'))
    else:
        w = synthetic.frequencies(64)[1]
        zn, ze = gold_fl[f'syn_{model}/zn'][0], gold_fl[f'syn_{model}/zn_err'][0]
    pts = PTS[model]
    assert all(_leaves_range(model, t, w) for t in pts)
    inv = BatchInversion(model, w, zn[None], ze[None], nwalkers=W, nsteps=T, seed=41, spectrum_offset=3)
    p0 = inv.draw_p0(0, 1)
    p0[0, 1:1 + len(pts)] = pts
    p0[0, W - len(pts):] = pts[::-1]
    prob = oracle.Problem(model, w, zn, ze, inv.param_bounds)
    dev = inv.device
    args = (_lib.dev_f64(w, dev), _lib.dev_f64(zn[None], dev), _lib.dev_f64(ze[None], dev),
            _lib.dev_f64(inv.param_bounds, dev))
    lp0 = engine.ensemble_run(inv._spec(), _lib.dev_f64(p0, dev), *args, nsteps=0, seed=41, spectrum0=3)['lp'].cpu().numpy()[0]
    want0 = prob.log_probability(p0[0])
    assert np.all(np.isfinite(want0)) and lp_err(lp0, want0).max() <= 1e-12
    res = inv.fit(p0=p0, keep_chain=True)
    ref = prob.run(p0[0], T, seed=41, spectrum=3)
    assert res['flags'][0] == 0 and not ref['nan']
    np.testing.assert_array_equal(res['chain'][0], ref['chain'])
    fin = np.isfinite(ref['log_prob'])
    assert np.array_equal(fin, np.isfinite(res['log_prob'][0]))
    assert lp_err(res['log_prob'][0][fin], ref['log_prob'][fin]).max() <= 1e-12
