"""WAIC of every spectrum inside batch and sharded fits (`bisip_waic`, `engine.waic`, `fit(..., waic=True)`,
`Inversion.get_waic`): parity with a NumPy restatement of the definitions over Z from the CPU oracle, the identity and
NaN cases, independence from sub-batching / keep_chain / the fit entry point, unchanged other keys, one launch per
sub-batch, and model selection on synthetic decomposition spectra."""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.special import logsumexp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ('elpd_waic', 'p_waic', 'se_elpd_waic', 'waic_pointwise', 'waic_n_high_p')


def _ref_waic(Z, y, yerr):
    """The definitions, in NumPy: Z (n, 2, N), y, yerr (2, N)."""
    s2 = yerr ** 2
    ll = -0.5 * np.sum((y - Z) ** 2 / s2 + 2 * np.log(s2), axis=1)         # (n, N): one data point per frequency
    n, N = ll.shape
    lppd = logsumexp(ll, axis=0) - np.log(n)
    p = np.var(ll, axis=0, ddof=1)
    elpd = lppd - p
    return dict(lppd=lppd, p=p, elpd=elpd.sum(), p_waic=p.sum(), se=np.sqrt(N * np.var(elpd, ddof=1)),
                n_high_p=int(np.count_nonzero(p > 0.4)))


def _close(got, ref, what):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
    assert np.all(err <= 1e-9), f"{what}: worst {err.max():.3e}"


def _check(out, b, ref):
    for k in ('lppd', 'p'):
        _close(out[k][b].cpu().numpy(), ref[k], k)
    for k in ('elpd', 'p_waic', 'se'):
        _close(out[k][b].item(), ref[k], k)
    assert not np.any(np.abs(ref['p'] - 0.4) < 1e-6), "p[j] too close to 0.4 for an exact count"
    assert int(out['n_high_p'][b].item()) == ref['n_high_p']


def _problem(model, w, y, ye, poly_deg=4, n_modes=1, n_tau=20, c_exp=1.0):
    from bisip_b200.batch import default_bounds, tau_grid
    from oracle import oracle
    _, bounds = default_bounds(model, poly_deg, n_modes)
    kw = {}
    if model == 'decomp':
        _, taus, lts = tau_grid(w, n_tau, poly_deg)
        kw = dict(taus=taus, log_taus=lts, c_exp=c_exp)
    return oracle.Problem(model, w, y, ye, bounds, n_modes=n_modes, **kw), bounds


def _spec(model, w, poly_deg=4, n_modes=1, n_tau=20, c_exp=1.0, precision='fp64'):
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
                            c_exp=float(c_exp), precision=_lib.PRECISIONS[precision])


def _data(model, B, N, seed, **kw):
    """Spectra from a parameter vector in the middle of the box, 2 % noise."""
    from bisip_b200.batch import default_bounds
    rng = np.random.default_rng(seed)
    w = 2 * np.pi * np.logspace(4, -2, N)
    _, bounds = default_bounds(model, kw.get('poly_deg', 4), kw.get('n_modes', 1))
    ys, yes = [], []
    for b in range(B):
        prob, _ = _problem(model, w, np.ones((2, N)), np.ones((2, N)), **kw)
        mid = 0.5 * (bounds[0] + bounds[1]) + 0.2 * (bounds[1] - bounds[0]) * rng.uniform(-1, 1, bounds.shape[1])
        z = prob.forward(mid)
        ye = 0.02 * np.abs(z) + 1e-3
        ys.append(z + ye * rng.standard_normal(z.shape))
        yes.append(ye)
    return w, np.array(ys), np.array(yes), bounds


def _run(model, theta, w, y, ye, per_spectrum=False, **kw):
    """engine.waic against the NumPy restatement for every spectrum.  theta (B, n, ndim)."""
    from bisip_b200 import _lib, engine
    dev = _lib.require_cuda()
    B = theta.shape[0]
    wb = np.stack([w * (1 + 0.03 * b) for b in range(B)]) if per_spectrum else w
    out = engine.waic(_spec(model, wb, **kw), _lib.dev_f64(theta, dev), _lib.dev_f64(wb, dev), _lib.dev_f64(y, dev),
                      _lib.dev_f64(ye, dev))
    for b in range(B):
        prob, _ = _problem(model, wb[b] if per_spectrum else w, y[b], ye[b], **kw)
        _check(out, b, _ref_waic(prob.forward(theta[b]), y[b], ye[b]))
    return out


def _uniform(bounds, B, n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(bounds[0], bounds[1], (B, n, bounds.shape[1]))


def _uniform_decomp(w, poly_deg, n_tau, B, n, seed):
    """Uniform draws for a decomposition: r0 in its box, coefficient a_i in [-1, 1] / L^i with L = max |log10 tau|,
    so that every term a_i log10(tau)^i of the RTD is at most 1.  With the default box, a_20 log10(tau)^20 reaches 1e15 at
    L = 6 and the sums cancel: any two FP64 evaluations of Z (two-stage, collapsed) then differ far above 1e-9."""
    from bisip_b200.batch import default_bounds, tau_grid
    _, bounds = default_bounds('decomp', poly_deg)
    L = np.abs(tau_grid(w, n_tau, poly_deg)[0]).max()
    th = _uniform(bounds, B, n, seed)
    th[..., 1:] /= L ** np.arange(poly_deg + 1)
    return th


DECOMP_CASES = [(pd, c) for pd in (0, 4, 9, 20) for c in (1.0, 0.5)]


@pytest.mark.parametrize('poly_deg,c_exp', DECOMP_CASES)
@pytest.mark.parametrize('per_spectrum', [False, True])
def test_waic_decomp_uniform_draws(poly_deg, c_exp, per_spectrum):
    kw = dict(poly_deg=poly_deg, n_tau=20, c_exp=c_exp)
    w, y, ye, bounds = _data('decomp', 2, 16, 3 + poly_deg, **kw)
    th = _uniform(bounds, 2, 300, poly_deg) if poly_deg < 20 else _uniform_decomp(w, poly_deg, 20, 2, 300, 20)
    _run('decomp', th, w, y, ye, per_spectrum=per_spectrum, **kw)


@pytest.mark.parametrize('model,kw', [('colecole', dict(n_modes=1)), ('colecole', dict(n_modes=2)),
                                      ('colecole', dict(n_modes=5)), ('dias', {}), ('shin', {})])
@pytest.mark.parametrize('per_spectrum', [False, True])
def test_waic_vector_models_uniform_draws(model, kw, per_spectrum):
    w, y, ye, bounds = _data(model, 3, 16, 5, **kw)
    _run(model, _uniform(bounds, 3, 500, 6), w, y, ye, per_spectrum=per_spectrum, **kw)


@pytest.mark.parametrize('n', [2, 25600, 40000])
def test_waic_chain_lengths(n):
    """n = 2 (the smallest), 25,600 and 40,000 (past what one CTA's shared memory would hold): the kernel has no
    length limit.  Draws near the data's parameter vector, so |ll| is moderate and p[j] is O(1)."""
    kw = dict(poly_deg=4, n_tau=20)
    w, y, ye, bounds = _data('decomp', 2, 16, 8, **kw)
    rng = np.random.default_rng(n)
    mid = 0.5 * (bounds[0] + bounds[1])
    th = mid + 0.02 * (bounds[1] - bounds[0]) * rng.standard_normal((2, n, bounds.shape[1]))
    _run('decomp', th, w, y, ye, **kw)


@pytest.mark.parametrize('model,kw', [('decomp', dict(poly_deg=4, n_tau=20)), ('colecole', dict(n_modes=2)),
                                      ('dias', {}), ('shin', {})])
def test_waic_on_fit_chains(model, kw):
    """Chains of short fits: the posterior's own spread."""
    import bisip_b200 as bb
    w, y, ye, _ = _data(model, 2, 16, 12, **kw)
    inv = bb.BatchInversion(model, w, y, ye, nwalkers=32, nsteps=300, seed=3, **kw)
    res = inv.fit(discard=150, thin=2, keep_chain=True)
    flat = res['chain'].reshape(2, -1, inv.ndim)
    _run(model, flat, w, y, ye, **kw)


def test_waic_identity():
    """Two identical samples: p == 0 exactly, and sum_j lppd[j] is the log-likelihood of that sample, which is the
    log-probability inside the box."""
    from bisip_b200 import _lib, engine
    kw = dict(poly_deg=4, n_tau=20)
    w, y, ye, bounds = _data('decomp', 2, 16, 21, **kw)
    dev = _lib.require_cuda()
    th0 = _uniform(bounds, 2, 1, 22)
    th = np.repeat(th0, 2, axis=1)
    spec = _spec('decomp', w, **kw)
    out = engine.waic(spec, _lib.dev_f64(th, dev), _lib.dev_f64(w, dev), _lib.dev_f64(y, dev), _lib.dev_f64(ye, dev))
    assert np.all(out['p'].cpu().numpy() == 0.0)
    assert np.all(out['p_waic'].cpu().numpy() == 0.0)
    lp = engine.log_probability(spec, _lib.dev_f64(th0, dev), _lib.dev_f64(w, dev), _lib.dev_f64(y, dev),
                                _lib.dev_f64(ye, dev), _lib.dev_f64(bounds, dev)).cpu().numpy()[:, 0]
    s = out['lppd'].cpu().numpy().sum(1)
    assert np.all(np.abs(s - lp) <= 1e-12 * np.abs(lp)), (s, lp)
    np.testing.assert_allclose(out['elpd'].cpu().numpy(), s, rtol=1e-14)              # elpd = sum_j lppd when p = 0


def test_waic_nan_sample():
    from bisip_b200 import _lib, engine
    kw = dict(poly_deg=4, n_tau=20)
    w, y, ye, bounds = _data('decomp', 3, 16, 31, **kw)
    dev = _lib.require_cuda()
    th = _uniform(bounds, 3, 400, 32)
    th[1, 123, 3] = np.nan
    spec = _spec('decomp', w, **kw)
    args = lambda t, yy, ee: (spec, _lib.dev_f64(t, dev), _lib.dev_f64(w, dev), _lib.dev_f64(yy, dev),
                              _lib.dev_f64(ee, dev))
    out = {k: v.cpu().numpy() for k, v in engine.waic(*args(th, y, ye)).items()}
    for k in ('lppd', 'p', 'elpd', 'p_waic', 'se'):
        assert np.all(np.isnan(out[k][1])), k
    assert out['n_high_p'][1] == 0
    keep = [0, 2]
    ref = {k: v.cpu().numpy() for k, v in engine.waic(*args(th[keep], y[keep], ye[keep])).items()}
    for k in out:
        np.testing.assert_array_equal(out[k][keep], ref[k], err_msg=k)
        assert not np.any(np.isnan(ref[k])), k


FIT_CASES = {
    'decomp-fp64': ('decomp', dict(poly_deg=4, n_tau=20, precision='fp64')),
    'decomp-collapsed': ('decomp', dict(poly_deg=4, n_tau=20, precision='fp64-collapsed')),
    'decomp-3xtf32': ('decomp', dict(poly_deg=4, n_tau=20, precision='3xtf32')),
    'colecole2': ('colecole', dict(n_modes=2)),
    'dias': ('dias', {}),
    'shin': ('shin', {}),
}


@pytest.mark.parametrize('case', sorted(FIT_CASES))
def test_fit_waic(case):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    model, kw = FIT_CASES[case]
    B = 4
    w, y, ye, _ = _data(model, B, 16, 41, **{k: v for k, v in kw.items() if k != 'precision'})
    ctor = dict(nwalkers=32, nsteps=300, seed=17, **kw)
    inv = bb.BatchInversion(model, w, y, ye, **ctor)
    fit = lambda **k: inv.fit(discard=100, thin=2, **k)
    full = fit(keep_chain=True, waic=True)
    N = y.shape[-1]
    assert full['elpd_waic'].shape == (B,) and full['waic_pointwise'].shape == (B, N)
    assert full['waic_n_high_p'].dtype == np.int32
    # the keys are engine.waic of the kept chain, bit for bit
    dev = inv.device
    ref = engine.waic(inv._spec(), _lib.dev_f64(full['chain'].reshape(B, -1, inv.ndim), dev), _lib.dev_f64(w, dev),
                      _lib.dev_f64(y, dev), _lib.dev_f64(ye, dev))
    ref = {k: v.cpu().numpy() for k, v in ref.items()}
    np.testing.assert_array_equal(full['elpd_waic'], ref['elpd'])
    np.testing.assert_array_equal(full['p_waic'], ref['p_waic'])
    np.testing.assert_array_equal(full['se_elpd_waic'], ref['se'])
    np.testing.assert_array_equal(full['waic_pointwise'], ref['lppd'] - ref['p'])
    np.testing.assert_array_equal(full['waic_n_high_p'], ref['n_high_p'])
    # every other key is bit-identical without waic
    plain = fit(keep_chain=True)
    assert set(full) == set(plain) | set(KEYS)
    for k in plain:
        np.testing.assert_array_equal(full[k], plain[k], err_msg=k)
    # the WAIC does not depend on how the fit was run
    runs = [fit(waic=True, batch_size=bs) for bs in (1, 3, B)]
    runs.append(fit(waic=True))
    runs.append(inv.fit_gathered(B, discard=100, thin=2, waic=True))
    runs.append(bb.fit_sharded(model, w, y, ye, discard=100, thin=2, waic=True, **ctor))
    for r in runs:
        for k in KEYS + tuple(plain.keys() - {'chain', 'log_prob'}):
            np.testing.assert_array_equal(r[k], full[k], err_msg=k)
    # one launch per sub-batch
    n0 = _lib.launch_count()
    fit(batch_size=3)
    base = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    fit(batch_size=3, waic=True)
    assert _lib.launch_count() - n0 - base == 2


def test_get_waic_equals_engine_on_a_data_file(data_files):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    m = bb.PolynomialDecomposition(data_files['SIP-K389175'], nwalkers=32, poly_deg=4, nsteps=400, seed=4)
    m.fit()
    flat = m.get_chain(discard=200, thin=2, flat=True)
    got = m.get_waic(chain=flat)
    again = m.get_waic(discard=200, thin=2)                       # parse_chain's other form, the same samples
    np.testing.assert_array_equal(again['waic_pointwise'], got['waic_pointwise'])
    assert again['elpd_waic'] == got['elpd_waic']
    dev = _lib.require_cuda()
    ref = engine.waic(m._spec(dev), _lib.dev_f64(flat[None], dev), _lib.dev_f64(m.data['w'], dev),
                      _lib.dev_f64(m.data['zn'][None], dev), _lib.dev_f64(m.data['zn_err'][None], dev))
    ref = {k: v[0].cpu().numpy() for k, v in ref.items()}
    assert got['elpd_waic'] == ref['elpd'] and got['p_waic'] == ref['p_waic'] and got['se_elpd_waic'] == ref['se']
    assert got['waic_n_high_p'] == ref['n_high_p']
    assert got['waic_pointwise'].shape == (m.data['w'].shape[0],)
    np.testing.assert_array_equal(got['waic_pointwise'], ref['lppd'] - ref['p'])


def test_waic_prefers_the_generating_model():
    """Synthetic spectra drawn from a 4th-degree decomposition: poly_deg 4 predicts them better than poly_deg 0, by
    more than two standard errors, for at least 95 % of the spectra."""
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    from bisip_b200.products import compare_waic
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
        res[pd] = inv.fit(discard=1000, thin=5, waic=True)
    c = compare_waic(res[4], res[0])
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
from test_gpu_waic import _data, KEYS
w, y, ye, _ = _data("decomp", 7, 16, 51, poly_deg=4, n_tau=20)
kw = dict(nwalkers=32, nsteps=300, seed=11, poly_deg=4, n_tau=20)
res = bb.fit_sharded("decomp", w, y, ye, discard=100, thin=2, waic=True, **kw)
ref = bb.BatchInversion("decomp", w, y, ye, **kw).fit(discard=100, thin=2, waic=True)
for k in KEYS + ("percentiles", "mean", "std", "acceptance_fraction", "flags"):
    np.testing.assert_array_equal(res[k], ref[k])            # independent of the number of ranks
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_waic_two_ranks_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker_waic.py"
    script.write_text(_NCCL_WORKER)
    port = str(29590 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out
        assert "ok" in out
