"""PSIS-LOO of every spectrum inside batch and sharded fits (`bisip_psis_loo`, `engine.psis_loo`, `fit(..., loo=True)`,
`Inversion.get_loo`): parity with the NumPy restatement `_ref_psis_loo` over Z from the CPU oracle, the chain lengths of
both kernel paths, the identity and NaN cases, a brute-force leave-one-out check, independence from sub-batching / the
fit entry point, unchanged other keys, two launches per sub-batch, and model selection on synthetic spectra."""
import os
import subprocess
import sys

import numpy as np
import pytest

from test_loo_host import _ref_psis_loo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ('elpd_loo', 'p_loo', 'se_elpd_loo', 'loo_pointwise', 'pareto_k', 'loo_n_high_k')


def _problem(model, w, y, ye, poly_deg=4, n_modes=1, n_tau=20, c_exp=1.0):
    from bisip_b200.batch import default_bounds, tau_grid
    from oracle import oracle
    _, bounds = default_bounds(model, poly_deg, n_modes)
    kw = {}
    if model == 'decomp':
        _, taus, lts = tau_grid(w, n_tau, poly_deg)
        kw = dict(taus=taus, log_taus=lts, c_exp=c_exp)
    return oracle.Problem(model, w, y, ye, bounds, n_modes=n_modes, **kw), bounds


def _spec(model, w, poly_deg=4, n_modes=1, n_tau=20, c_exp=1.0):
    """ModelSpec on the device; w (N,) or (B, N) gives shared or per-spectrum tau grids."""
    from bisip_b200 import _lib, engine
    from bisip_b200.batch import _MODEL_IDS, default_bounds, tau_grid
    dev = _lib.require_cuda()
    names, _ = default_bounds(model, poly_deg, n_modes)
    taus = lts = None
    if model == 'decomp':
        _, t, l = tau_grid(w, n_tau, poly_deg)
        taus, lts = _lib.dev_f64(t, dev), _lib.dev_f64(l, dev)
    return engine.ModelSpec(model=_MODEL_IDS[model], ndim=len(names), n_modes=n_modes, taus=taus, log_taus=lts,
                            c_exp=float(c_exp), precision=_lib.PREC_FP64)


def _draws(model, spreads, n, seed, N=16, per_spectrum=False, **kw):
    """One spectrum per spread: data from a parameter vector near the middle of the box (2 % noise), and n draws
    Gaussian around that vector with standard deviation `spread` x the box width, clipped into the box.  For the
    decomposition the width of coefficient a_i is divided by L^i, L = max |log10 tau|, so that every draw keeps the
    terms a_i log10(tau)^i of the RTD moderate (in the full box two FP64 evaluations of Z at poly_deg 20 disagree far
    above 1e-9).  Returns theta (B, n, ndim), w (N,) or (B, N), y, yerr (B, 2, N) and the ll of every draw from the
    oracle's Z (B, n, N)."""
    from bisip_b200.batch import tau_grid
    rng = np.random.default_rng(seed)
    B = len(spreads)
    w0 = 2 * np.pi * np.logspace(4, -2, N)
    ws = np.stack([w0 * (1 + 0.03 * b) for b in range(B)]) if per_spectrum else np.stack([w0] * B)
    ths, ys, yes, lls = [], [], [], []
    for b, s in enumerate(spreads):
        prob, bounds = _problem(model, ws[b], np.ones((2, N)), np.ones((2, N)), **kw)
        width = bounds[1] - bounds[0]
        if model == 'decomp':
            pd = kw.get('poly_deg', 4)
            width = width.copy()
            width[1:] /= np.abs(tau_grid(ws[b], kw.get('n_tau', 20), pd)[0]).max() ** np.arange(pd + 1)
        c = 0.5 * (bounds[0] + bounds[1]) + 0.2 * width * rng.uniform(-1, 1, bounds.shape[1])
        z = prob.forward(c)
        ye = 0.02 * np.abs(z) + 1e-3
        y = z + ye * rng.standard_normal(z.shape)
        th = np.clip(c + s * width * rng.standard_normal((n, bounds.shape[1])), bounds[0], bounds[1])
        Z = _problem(model, ws[b], y, ye, **kw)[0].forward(th)
        s2 = ye ** 2
        lls.append(-0.5 * np.sum((y - Z) ** 2 / s2 + 2 * np.log(s2), axis=1))
        ths.append(th), ys.append(y), yes.append(ye)
    return np.array(ths), (ws if per_spectrum else w0), np.array(ys), np.array(yes), np.array(lls)


def _close(got, ref, what):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    same_inf = np.isinf(ref) & (got == ref)
    err = np.where(same_inf, 0.0, np.abs(got - ref) / np.maximum(1.0, np.abs(ref)))
    assert np.all(err <= 1e-9), f"{what}: worst {np.nanmax(err):.3e}"


def _check(out, b, ref):
    """One spectrum of engine.psis_loo against the reference; the reference's tail sets and k must be unambiguous."""
    assert np.all(ref['gap'] > 1e-6), "the M-th and (M+1)-th largest log-ratios are too close for an exact tail set"
    assert not np.any(np.abs(ref['pareto_k'] - ref['threshold']) < 1e-6), "k too close to the threshold"
    for k in ('elpd_i', 'p_i', 'pareto_k'):
        _close(out[k][b].cpu().numpy(), ref[k], k)
    for k in ('elpd', 'p_loo', 'se'):
        _close(out[k][b].item(), ref[k], k)
    assert int(out['n_high_k'][b].item()) == ref['n_high_k']


def _run(model, spreads, n, seed, per_spectrum=False, **kw):
    from bisip_b200 import _lib, engine
    dev = _lib.require_cuda()
    th, w, y, ye, ll = _draws(model, spreads, n, seed, per_spectrum=per_spectrum, **kw)
    out = engine.psis_loo(_spec(model, w, **kw), _lib.dev_f64(th, dev), _lib.dev_f64(w, dev), _lib.dev_f64(y, dev),
                          _lib.dev_f64(ye, dev))
    refs = [_ref_psis_loo(ll[b]) for b in range(len(spreads))]
    for b, ref in enumerate(refs):
        _check(out, b, ref)
    return out, refs


DECOMP_SPREADS, VECTOR_SPREADS = (0.0003, 0.001, 0.002), (0.001, 0.003, 0.01)
PARITY_CASES = ([('decomp', dict(poly_deg=pd, c_exp=c)) for pd in (0, 4, 9, 20) for c in (1.0, 0.5)] +
                [('colecole', dict(n_modes=1)), ('colecole', dict(n_modes=2)), ('colecole', dict(n_modes=5)),
                 ('dias', {}), ('shin', {})])


# seeds of the cases whose default seed 100 + i gives a reference with a near-tie at the cutoff
PARITY_SEEDS = {11: 310, 12: 320}


def _parity_args(i, per_spectrum):
    model, kw = PARITY_CASES[i]
    return (model, (DECOMP_SPREADS if model == 'decomp' else VECTOR_SPREADS), 2000, PARITY_SEEDS.get(i, 100 + i),
            per_spectrum, kw)


@pytest.mark.parametrize('i', range(len(PARITY_CASES)))
@pytest.mark.parametrize('per_spectrum', [False, True])
def test_psis_loo_parity(i, per_spectrum):
    model, spreads, n, seed, ps, kw = _parity_args(i, per_spectrum)
    _run(model, spreads, n, seed, per_spectrum=ps, **kw)


def test_psis_loo_parity_covers_every_k_band():
    """The parity cases' references hold k < 0.5, 0.5 < k < 0.7 and k > 0.7, and a frequency whose smoothed tail was
    truncated at 0 (CPU only: the same inputs as test_psis_loo_parity)."""
    ks, trunc = [], 0
    for i in range(len(PARITY_CASES)):
        for per_spectrum in (False, True):
            model, spreads, n, seed, ps, kw = _parity_args(i, per_spectrum)
            ll = _draws(model, spreads, n, seed, per_spectrum=ps, **kw)[4]
            for b in range(len(spreads)):
                r = _ref_psis_loo(ll[b])
                ks.append(r['pareto_k'])
                trunc += int(r['truncated'].sum())
    k = np.concatenate(ks)
    bands = {'k<0.5': np.sum(k < 0.5), '0.5<k<0.7': np.sum((k > 0.5) & (k < 0.7)), 'k>0.7': np.sum(k > 0.7)}
    print('parity k bands', bands, 'truncated', trunc)
    assert all(v > 0 for v in bands.values()), bands
    assert trunc > 0


@pytest.mark.parametrize('n', [2, 20, 25600, 40000])
def test_psis_loo_chain_lengths(n):
    """n = 2 and 20 (M <= 4: k = inf), 25,600 (the C5 chain, shared-memory path) and 40,000 (past one CTA's shared
    memory: the column is recomputed per pass)."""
    out, refs = _run('decomp', (0.0003, 0.001), n, n, poly_deg=4, n_tau=20)
    if n <= 20:
        assert np.all(np.isinf(out['pareto_k'].cpu().numpy()))
    else:
        assert all(np.all(np.isfinite(r['pareto_k'])) for r in refs)


def test_psis_loo_identity():
    """Two equal samples: an empty tail, k = inf, elpd_loo_j = lppd_j (bisip_waic's) and p_loo = 0 exactly."""
    from bisip_b200 import _lib, engine
    dev = _lib.require_cuda()
    th, w, y, ye, _ = _draws('decomp', (0.001, 0.001), 1, 21, poly_deg=4)
    th = np.repeat(th, 2, axis=1)
    args = (_spec('decomp', w, poly_deg=4), _lib.dev_f64(th, dev), _lib.dev_f64(w, dev), _lib.dev_f64(y, dev),
            _lib.dev_f64(ye, dev))
    out = {k: v.cpu().numpy() for k, v in engine.psis_loo(*args).items()}
    wa = engine.waic(*args)
    assert np.all(np.isinf(out['pareto_k']))
    np.testing.assert_array_equal(out['elpd_i'], wa['lppd'].cpu().numpy())
    assert np.all(out['p_i'] == 0.0) and np.all(out['p_loo'] == 0.0)


def test_psis_loo_nan_sample():
    from bisip_b200 import _lib, engine
    dev = _lib.require_cuda()
    th, w, y, ye, _ = _draws('decomp', (0.001, 0.001, 0.002), 400, 31, poly_deg=4)
    th[1, 123, 3] = np.nan
    spec = _spec('decomp', w, poly_deg=4)
    args = lambda t, yy, ee: (spec, _lib.dev_f64(t, dev), _lib.dev_f64(w, dev), _lib.dev_f64(yy, dev),
                              _lib.dev_f64(ee, dev))
    out = {k: v.cpu().numpy() for k, v in engine.psis_loo(*args(th, y, ye)).items()}
    for k in ('elpd_i', 'p_i', 'pareto_k', 'elpd', 'p_loo', 'se'):
        assert np.all(np.isnan(out[k][1])), k
    assert out['n_high_k'][1] == 0
    keep = [0, 2]
    ref = {k: v.cpu().numpy() for k, v in engine.psis_loo(*args(th[keep], y[keep], ye[keep])).items()}
    for k in out:
        np.testing.assert_array_equal(out[k][keep], ref[k], err_msg=k)
        assert not np.any(np.isnan(ref[k])), k


def test_psis_loo_matches_brute_force_leave_one_out():
    """One synthetic decomposition spectrum with 16 frequencies, fitted 17 times in one batch: copy j < 16 with
    zn_err[:, j] = 1e100, which makes frequency j's term a constant and so removes it from the posterior, copy 16 with
    the full data.  The exact leave-one-out predictive density of frequency j is lppd_j over copy j's chain with the
    original errors; PSIS-LOO of copy 16 must agree with it within 0.1 nats wherever k < 0.5."""
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    N = 16
    _, w = synthetic.frequencies(N)
    probe = BatchInversion('decomp', w, np.zeros((1, 2, N)), np.ones((1, 2, N)), poly_deg=4)
    fwd = lambda th, ww: engine.forward(probe._spec(), _lib.dev_f64(th[:, None, :], probe.device),
                                        _lib.dev_f64(ww, probe.device))[:, 0].cpu().numpy()
    syn = synthetic.make('decomp', 3, 4, fwd, N=N, poly_deg=4)
    zn = np.repeat(syn['zn'], N + 1, axis=0)
    err = np.repeat(syn['zn_err'], N + 1, axis=0)
    for j in range(N):
        err[j, :, j] = 1e100
    inv = bb.BatchInversion('decomp', syn['w'], zn, err, nwalkers=64, nsteps=3000, seed=5, poly_deg=4)
    res = inv.fit(discard=1000, thin=10, keep_chain=True, loo=True)
    dev = inv.device
    flat = res['chain'].reshape(N + 1, -1, inv.ndim)
    wa = engine.waic(inv._spec(), _lib.dev_f64(flat[:N], dev), _lib.dev_f64(syn['w'], dev),
                     _lib.dev_f64(np.repeat(syn['zn'], N, axis=0), dev),
                     _lib.dev_f64(np.repeat(syn['zn_err'], N, axis=0), dev))
    exact = np.diag(wa['lppd'].cpu().numpy())
    k = res['pareto_k'][N]
    good = k < 0.5
    dev_max = np.max(np.abs(res['loo_pointwise'][N][good] - exact[good]))
    print(f'brute-force LOO: {int(good.sum())} of {N} frequencies with k < 0.5, max |psis - exact| = {dev_max:.4f} nats')
    assert good.sum() >= N // 2, k
    assert dev_max <= 0.1, (res['loo_pointwise'][N], exact, k)


FIT_CASES = {
    'decomp-fp64': ('decomp', dict(poly_deg=4, n_tau=20, precision='fp64')),
    'decomp-collapsed': ('decomp', dict(poly_deg=4, n_tau=20, precision='fp64-collapsed')),
    'decomp-3xtf32': ('decomp', dict(poly_deg=4, n_tau=20, precision='3xtf32')),
    'colecole2': ('colecole', dict(n_modes=2)),
    'dias': ('dias', {}),
    'shin': ('shin', {}),
}


def _fit_data(model, B, seed, **kw):
    _, w, y, ye, _ = _draws(model, (0.001,) * B, 1, seed, **kw)
    return w, y, ye


@pytest.mark.parametrize('case', sorted(FIT_CASES))
def test_fit_loo(case):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    model, kw = FIT_CASES[case]
    B = 4
    w, y, ye = _fit_data(model, B, 41, **{k: v for k, v in kw.items() if k != 'precision'})
    ctor = dict(nwalkers=32, nsteps=300, seed=17, **kw)
    inv = bb.BatchInversion(model, w, y, ye, **ctor)
    fit = lambda **k: inv.fit(discard=100, thin=2, **k)
    full = fit(keep_chain=True, loo=True)
    N = y.shape[-1]
    assert full['elpd_loo'].shape == (B,) and full['loo_pointwise'].shape == (B, N)
    assert full['pareto_k'].shape == (B, N) and full['loo_n_high_k'].dtype == np.int32
    # the keys are engine.psis_loo of the kept chain, bit for bit
    dev = inv.device
    ref = engine.psis_loo(inv._spec(), _lib.dev_f64(full['chain'].reshape(B, -1, inv.ndim), dev), _lib.dev_f64(w, dev),
                          _lib.dev_f64(y, dev), _lib.dev_f64(ye, dev))
    ref = {k: v.cpu().numpy() for k, v in ref.items()}
    for key, rk in (('elpd_loo', 'elpd'), ('p_loo', 'p_loo'), ('se_elpd_loo', 'se'), ('loo_pointwise', 'elpd_i'),
                    ('pareto_k', 'pareto_k'), ('loo_n_high_k', 'n_high_k')):
        np.testing.assert_array_equal(full[key], ref[rk], err_msg=key)
    # every other key is bit-identical without loo
    plain = fit(keep_chain=True)
    assert set(full) == set(plain) | set(KEYS)
    for k in plain:
        np.testing.assert_array_equal(full[k], plain[k], err_msg=k)
    # PSIS-LOO does not depend on how the fit was run
    runs = [fit(loo=True, batch_size=bs) for bs in (1, 3, B)]
    runs.append(inv.fit_gathered(B, discard=100, thin=2, loo=True))
    runs.append(bb.fit_sharded(model, w, y, ye, discard=100, thin=2, loo=True, **ctor))
    for r in runs:
        for k in KEYS + tuple(plain.keys() - {'chain', 'log_prob'}):
            np.testing.assert_array_equal(r[k], full[k], err_msg=k)
    # two launches per sub-batch
    n0 = _lib.launch_count()
    fit(batch_size=3)
    base = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    fit(batch_size=3, loo=True)
    assert _lib.launch_count() - n0 - base == 4


def test_get_loo_equals_engine_on_a_data_file(data_files):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    m = bb.PolynomialDecomposition(data_files['SIP-K389175'], nwalkers=32, poly_deg=4, nsteps=400, seed=4)
    m.fit()
    flat = m.get_chain(discard=200, thin=2, flat=True)
    got = m.get_loo(chain=flat)
    again = m.get_loo(discard=200, thin=2)                        # parse_chain's other form, the same samples
    np.testing.assert_array_equal(again['loo_pointwise'], got['loo_pointwise'])
    np.testing.assert_array_equal(again['pareto_k'], got['pareto_k'])
    dev = _lib.require_cuda()
    ref = engine.psis_loo(m._spec(dev), _lib.dev_f64(flat[None], dev), _lib.dev_f64(m.data['w'], dev),
                          _lib.dev_f64(m.data['zn'][None], dev), _lib.dev_f64(m.data['zn_err'][None], dev))
    ref = {k: v[0].cpu().numpy() for k, v in ref.items()}
    assert got['elpd_loo'] == ref['elpd'] and got['p_loo'] == ref['p_loo'] and got['se_elpd_loo'] == ref['se']
    assert got['loo_n_high_k'] == ref['n_high_k']
    assert got['loo_pointwise'].shape == (m.data['w'].shape[0],)
    np.testing.assert_array_equal(got['loo_pointwise'], ref['elpd_i'])
    np.testing.assert_array_equal(got['pareto_k'], ref['pareto_k'])


def test_loo_prefers_the_generating_model():
    """Synthetic spectra drawn from a 4th-degree decomposition: poly_deg 4 predicts them better than poly_deg 0, by
    more than two standard errors, for at least 95 % of the spectra."""
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    from bisip_b200.products import compare_loo
    B, N = 40, 32
    _, w = synthetic.frequencies(N)
    probe = BatchInversion('decomp', w, np.zeros((1, 2, N)), np.ones((1, 2, N)), poly_deg=4)
    fwd = lambda th, ww: engine.forward(probe._spec(), _lib.dev_f64(th[:, None, :], probe.device),
                                        _lib.dev_f64(ww, probe.device))[:, 0].cpu().numpy()
    syn = synthetic.make('decomp', 0, B, fwd, N=N, poly_deg=4)
    res = {}
    for pd in (0, 4):
        inv = bb.BatchInversion('decomp', syn['w'], syn['zn'], syn['zn_err'], nwalkers=32, nsteps=2000, seed=7,
                                poly_deg=pd)
        res[pd] = inv.fit(discard=1000, thin=5, loo=True)
    c = compare_loo(res[4], res[0])
    better = (c['elpd_diff'] > 2 * c['se_diff'])
    assert np.count_nonzero(better) >= 0.95 * B, (c['elpd_diff'], c['se_diff'])


_NCCL_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"]); sys.path.insert(0, os.path.join(os.environ["BISIP_ROOT"], "tests"))
import numpy as np, torch, torch.distributed as dist
import bisip_b200 as bb
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=rank, world_size=world,
                        device_id=torch.device("cuda", rank))
from test_gpu_loo import _fit_data, KEYS
w, y, ye = _fit_data("decomp", 7, 51, poly_deg=4, n_tau=20)
kw = dict(nwalkers=32, nsteps=300, seed=11, poly_deg=4, n_tau=20)
res = bb.fit_sharded("decomp", w, y, ye, discard=100, thin=2, loo=True, **kw)
ref = bb.BatchInversion("decomp", w, y, ye, **kw).fit(discard=100, thin=2, loo=True)
for k in KEYS + ("percentiles", "mean", "std", "acceptance_fraction", "flags"):
    np.testing.assert_array_equal(res[k], ref[k])            # independent of the number of ranks
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_loo_two_ranks_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker_loo.py"
    script.write_text(_NCCL_WORKER)
    port = str(29300 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out
        assert "ok" in out
