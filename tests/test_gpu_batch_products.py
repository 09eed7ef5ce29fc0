"""RTD, total-chargeability and model-curve percentiles of every spectrum inside batch and sharded fits
(`bisip_rtd_stats`, `fit(..., rtd=True, model_curves=True)`, `PolynomialDecomposition.get_rtd(p=...)`): parity with
NumPy over the kept chain, independence from sub-batching / keep_chain / the fit entry point, unchanged other keys,
one launch per sub-batch and flag, both kernel paths, and the other models' model curves."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P3 = (2.5, 50, 97.5)
P20 = tuple(float(q) for q in np.linspace(1, 99, 20))
NEW_KEYS = ('rtd_percentiles', 'rtd_mean', 'rtd_std', 'total_chargeability_percentiles', 'total_chargeability_mean',
            'total_chargeability_std', 'model_percentiles')


def _dev(a):
    from bisip_b200 import _lib
    return _lib.dev_f64(a, _lib.require_cuda())


def _survey(model, B, N=16, **kw):
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    _, w = synthetic.frequencies(N)
    probe = BatchInversion(model, w, np.zeros((1, 2, N)), np.ones((1, 2, N)), **kw)
    fwd = lambda th, ww: engine.forward(probe._spec(), _lib.dev_f64(th[:, None, :], probe.device),
                                        _lib.dev_f64(ww, probe.device))[:, 0].cpu().numpy()
    extra = {k: kw[k] for k in ('poly_deg', 'n_tau', 'n_modes') if k in kw}
    return synthetic.make(model, 0, B, fwd, N=N, **extra)


def _bound(a, lt):
    """sum_l sum_i |a_i log_tau_l^i| per sample: the scale of the rounding of a total chargeability."""
    return np.abs(a) @ np.abs(lt).sum(-1)


def _check_rtd(flat, lt, p, pct, mean, std, tot_pct, tot_mean, tot_std):
    """One spectrum's products against NumPy over its flat chain (n, ndim)."""
    from bisip_b200.products import relaxation_time_distribution
    m = relaxation_time_distribution(flat[:, 1:], lt)
    np.testing.assert_array_equal(pct, np.percentile(m, p, axis=0))                      # bit for bit
    scale = np.abs(m).max()
    np.testing.assert_allclose(mean, m.mean(0), rtol=1e-13, atol=1e-13 * scale)
    np.testing.assert_allclose(std, m.std(0), rtol=1e-13, atol=1e-13 * scale)
    tot, tol = m.sum(-1), 1e-13 * _bound(flat[:, 1:], lt).max()
    np.testing.assert_allclose(tot_pct, np.percentile(tot, p), rtol=0, atol=tol)
    np.testing.assert_allclose(tot_mean, tot.mean(), rtol=0, atol=tol)
    np.testing.assert_allclose(tot_std, tot.std(), rtol=1e-12, atol=tol)


def _theta(B, n, n_coef, seed):
    rng = np.random.default_rng(seed)
    th = rng.uniform(-1, 1, (B, n, 1 + n_coef))
    th[..., 0] += 1.0
    return th


@pytest.mark.parametrize('n,n_coef,per_spectrum,p', [
    (3000, 5, False, P3), (3000, 10, True, P20), (500, 32, False, (0, 100)),
    (30000, 5, True, P3),          # 234 KB column: past one CTA's shared memory, the global-memory path
])
def test_rtd_stats_matches_numpy(n, n_coef, per_spectrum, p):
    from bisip_b200 import batch, engine, synthetic
    B, N = 3, 12
    w = synthetic.frequencies(N)[1] * (1 + 0.1 * np.arange(B)[:, None] if per_spectrum else 1)
    _, _, lt = batch.tau_grid(w, 2 * N, n_coef - 1)
    th = _theta(B, n, n_coef, seed=n + n_coef)
    got = engine.rtd_stats(_dev(th), _dev(lt), p=p, want_mean=True, want_std=True)
    pct, mean, std = (got[k].cpu().numpy() for k in ('pct', 'mean', 'std'))
    S = lt.shape[-1]
    assert pct.shape == (B, len(p), S + 1) and mean.shape == std.shape == (B, S + 1)
    for b in range(B):
        ltb = lt[b] if per_spectrum else lt
        _check_rtd(th[b], ltb, p, pct[b, :, :S], mean[b, :S], std[b, :S], pct[b, :, S], mean[b, S], std[b, S])
    # a spectrum's products depend on its own chain only; percentile-only and mean-only calls give the same values
    one = engine.rtd_stats(_dev(th[1:2]), _dev(lt[1:2] if per_spectrum else lt), p=p)
    np.testing.assert_array_equal(one['pct'].cpu().numpy()[0], pct[1])
    assert one['mean'] is None and one['std'] is None
    only = engine.rtd_stats(_dev(th), _dev(lt), want_mean=True)
    assert only['pct'] is None
    np.testing.assert_array_equal(only['mean'].cpu().numpy(), mean)


def test_rtd_stats_total_chargeability_per_sample():
    """With one sample per 'spectrum', the median is the sample's own value: the per-sample totals against NumPy."""
    from bisip_b200 import batch, engine, synthetic
    from bisip_b200.products import relaxation_time_distribution
    for n_coef in (5, 10):
        _, _, lt = batch.tau_grid(synthetic.frequencies(20)[1], 40, n_coef - 1)
        th = _theta(1, 4000, n_coef, seed=n_coef)[0]
        got = engine.rtd_stats(_dev(th[:, None, :]), _dev(lt), p=50)['pct'].cpu().numpy()[:, 0]
        m = relaxation_time_distribution(th[:, 1:], lt)
        np.testing.assert_array_equal(got[:, :-1], m)
        err = np.abs(got[:, -1] - m.sum(-1))
        assert np.all(err <= 1e-13 * _bound(th[:, 1:], lt)), err.max()


def test_rtd_stats_nan_sample():
    from bisip_b200 import batch, engine, synthetic
    _, _, lt = batch.tau_grid(synthetic.frequencies(10)[1], 20, 4)
    for n in (200, 30000):            # shared-memory and global-memory paths
        th = _theta(2, n, 5, seed=3)
        th[1, n // 3, 2] = np.nan
        got = engine.rtd_stats(_dev(th), _dev(lt), p=P3, want_mean=True)
        pct, mean = got['pct'].cpu().numpy(), got['mean'].cpu().numpy()
        assert np.all(np.isnan(pct[1])) and np.all(np.isnan(mean[1]))
        assert np.all(np.isfinite(pct[0])) and np.all(np.isfinite(mean[0]))


def test_get_rtd_past_shared_memory_equals_numpy(data_files):
    import bisip_b200 as bb
    from bisip_b200 import products
    m = bb.PolynomialDecomposition(data_files['SIP-K389175'], nwalkers=32, poly_deg=4, nsteps=10)
    flat = np.random.default_rng(5).uniform(*m.param_bounds, (31000, 6))
    for p in (P3, P20):
        want = np.percentile(products.relaxation_time_distribution(flat[:, 1:], m.log_taus), p, axis=0)
        np.testing.assert_array_equal(m.get_rtd(p=list(p), chain=flat), want)
    assert m.get_rtd(p=50, chain=flat[:500]).shape == (m.log_taus.shape[1],)


def _fit_all(inv, **kw):
    return inv.fit(discard=100, thin=2, **kw)


FIT_CASES = {
    'decomp-fp64': dict(poly_deg=4, n_tau=32),
    'decomp-collapsed-pd9': dict(poly_deg=9, n_tau=24),          # n_coef 10: the collapsed form
}


@pytest.mark.parametrize('case', sorted(FIT_CASES))
@pytest.mark.parametrize('per_spectrum', [False, True])
def test_fit_products(case, per_spectrum):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    kw = FIT_CASES[case]
    B = 5
    syn = _survey('decomp', B, **kw)
    w = syn['w'] * (1 + 0.05 * np.arange(B)[:, None]) if per_spectrum else syn['w']
    ctor = dict(nwalkers=32, nsteps=300, seed=23, **kw)
    inv = bb.BatchInversion('decomp', w, syn['zn'], syn['zn_err'], **ctor)
    p = P20 if per_spectrum else P3
    full = _fit_all(inv, percentiles=p, keep_chain=True, rtd=True, model_curves=True)
    S, N = inv.log_taus.shape[-1], syn['zn'].shape[-1]
    assert full['rtd_percentiles'].shape == (B, len(p), S) and full['rtd_mean'].shape == (B, S)
    assert full['total_chargeability_percentiles'].shape == (B, len(p)) and full['total_chargeability_std'].shape == (B,)
    assert full['model_percentiles'].shape == (B, len(p), 2, N)
    dev = inv.device
    m_mean, tot_of_mean = inv.rtd()                      # the RTD of the mean coefficients, on the host
    for b in range(B):
        flat = full['chain'][b].reshape(-1, inv.ndim)
        lt = inv.log_taus[b] if per_spectrum else inv.log_taus
        _check_rtd(flat, lt, p, full['rtd_percentiles'][b], full['rtd_mean'][b], full['rtd_std'][b],
                   full['total_chargeability_percentiles'][b], full['total_chargeability_mean'][b],
                   full['total_chargeability_std'][b])
        tol = 1e-12 * _bound(flat[:, 1:], lt).max()      # the mean is linear: equal up to rounding
        np.testing.assert_allclose(full['total_chargeability_mean'][b], tot_of_mean[b], rtol=1e-12, atol=tol)
        np.testing.assert_allclose(full['rtd_mean'][b], m_mean[b], rtol=1e-12, atol=tol)
        spec = inv._spec(b, b + 1) if per_spectrum else inv._spec()
        wb = _lib.dev_f64(w[b] if per_spectrum else w, dev)
        th = _lib.dev_f64(flat[None], dev)
        np.testing.assert_array_equal(full['model_percentiles'][b], engine.model_percentile(spec, th, wb, p)[0].cpu().numpy())
        Z = engine.forward(spec, th, wb)[0].cpu().numpy()                   # (n, 2, N)
        np.testing.assert_allclose(full['model_percentiles'][b], np.percentile(Z, p, axis=0), rtol=0, atol=1e-12)
    # every other key is bit-identical without the flags; the products do not depend on how the fit was run
    plain = _fit_all(inv, percentiles=p, keep_chain=True)
    assert set(full) == set(plain) | set(NEW_KEYS)
    for k in plain:
        np.testing.assert_array_equal(full[k], plain[k], err_msg=k)
    runs = [_fit_all(inv, percentiles=p, rtd=True, model_curves=True, batch_size=bs) for bs in (1, 2, B)]
    runs.append(inv.fit_gathered(B, discard=100, thin=2, percentiles=p, rtd=True, model_curves=True))
    runs.append(bb.fit_sharded('decomp', w, syn['zn'], syn['zn_err'], discard=100, thin=2, percentiles=p, rtd=True,
                               model_curves=True, **ctor))
    for r in runs:
        for k in NEW_KEYS + tuple(plain.keys() - {'chain', 'log_prob'}):
            np.testing.assert_array_equal(r[k], full[k], err_msg=k)
    # one launch per sub-batch and flag (per 16 percentiles)
    per_call = -(-len(p) // 16)
    n0 = _lib.launch_count()
    _fit_all(inv, percentiles=p, batch_size=3)
    base = _lib.launch_count() - n0
    for flags, extra in (({'rtd': True}, 2 * per_call), ({'model_curves': True}, 2 * per_call),
                         ({'rtd': True, 'model_curves': True}, 4 * per_call)):
        n0 = _lib.launch_count()
        _fit_all(inv, percentiles=p, batch_size=3, **flags)
        assert _lib.launch_count() - n0 - base == extra, flags


def test_fit_products_past_shared_memory():
    """64 walkers x 500 kept steps = 32,000 samples per spectrum: the RTD global-memory path and the model-curve
    fallback (forward + column statistics)."""
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    B = 2
    kw = dict(poly_deg=4, n_tau=32)
    syn = _survey('decomp', B, **kw)
    inv = bb.BatchInversion('decomp', syn['w'], syn['zn'], syn['zn_err'], nwalkers=64, nsteps=500, seed=5, **kw)
    res = inv.fit(keep_chain=True, rtd=True, model_curves=True)
    assert res['chain'].shape[1] * res['chain'].shape[2] == 32000
    dev = inv.device
    spec, w = inv._spec(), _lib.dev_f64(syn['w'], dev)
    for b in range(B):
        flat = res['chain'][b].reshape(-1, inv.ndim)
        _check_rtd(flat, inv.log_taus, P3, res['rtd_percentiles'][b], res['rtd_mean'][b], res['rtd_std'][b],
                   res['total_chargeability_percentiles'][b], res['total_chargeability_mean'][b],
                   res['total_chargeability_std'][b])
        Z = engine.forward(spec, _lib.dev_f64(flat[None], dev), w)[0].cpu().numpy()
        np.testing.assert_array_equal(res['model_percentiles'][b], np.percentile(Z, P3, axis=0))
    one = bb.BatchInversion('decomp', syn['w'], syn['zn'], syn['zn_err'], nwalkers=64, nsteps=500, seed=5, **kw)
    one.MODEL_CURVE_BYTES = 1                                    # one spectrum per fallback group
    again = one.fit(rtd=True, model_curves=True)
    for k in NEW_KEYS:
        np.testing.assert_array_equal(again[k], res[k], err_msg=k)


@pytest.mark.parametrize('model,kw', [('colecole', dict(n_modes=2)), ('dias', {}), ('shin', {})])
def test_model_curves_other_models(model, kw):
    import bisip_b200 as bb
    from bisip_b200 import _lib, engine
    B = 3
    syn = _survey(model, B, **kw)
    inv = bb.BatchInversion(model, syn['w'], syn['zn'], syn['zn_err'], nwalkers=32, nsteps=300, seed=9, **kw)
    n0 = _lib.launch_count()
    with pytest.raises(ValueError, match='decomp'):
        inv.fit(discard=100, rtd=True)
    assert _lib.launch_count() == n0                             # raised before anything was launched
    res = inv.fit(discard=100, thin=2, keep_chain=True, model_curves=True)
    assert res['model_percentiles'].shape == (B, 3, 2, syn['zn'].shape[-1])
    spec, w = inv._spec(), _lib.dev_f64(syn['w'], inv.device)
    for b in range(B):
        th = _lib.dev_f64(res['chain'][b].reshape(1, -1, inv.ndim), inv.device)
        np.testing.assert_array_equal(res['model_percentiles'][b], engine.model_percentile(spec, th, w, P3)[0].cpu().numpy())
        Z = engine.forward(spec, th, w)[0].cpu().numpy()
        np.testing.assert_allclose(res['model_percentiles'][b], np.percentile(Z, P3, axis=0), rtol=0, atol=1e-12)
    plain = inv.fit(discard=100, thin=2, keep_chain=True)
    for k in plain:
        np.testing.assert_array_equal(res[k], plain[k], err_msg=k)


def test_model_curves_equal_get_model_percentile_on_a_data_file(data_files):
    import bisip_b200 as bb
    path = data_files['SIP-K389175']
    inv = bb.BatchInversion.from_files('decomp', [path], nwalkers=32, nsteps=400, poly_deg=4, seed=4)
    res = inv.fit(discard=200, thin=2, keep_chain=True, model_curves=True, rtd=True)
    m = bb.PolynomialDecomposition(path, nwalkers=32, poly_deg=4, nsteps=400)
    flat = res['chain'][0].reshape(-1, 6)
    np.testing.assert_array_equal(res['model_percentiles'][0], m.get_model_percentile(list(P3), chain=flat))
    np.testing.assert_array_equal(res['rtd_percentiles'][0], m.get_rtd(p=list(P3), chain=flat))


_NCCL_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"]); sys.path.insert(0, os.path.join(os.environ["BISIP_ROOT"], "tests"))
import numpy as np, torch, torch.distributed as dist
import bisip_b200 as bb
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=rank, world_size=world,
                        device_id=torch.device("cuda", rank))
from test_gpu_batch_products import _survey, NEW_KEYS
kw = dict(nwalkers=32, nsteps=300, seed=11, poly_deg=4, n_tau=32)
syn = _survey("decomp", 7, poly_deg=4, n_tau=32)
res = bb.fit_sharded("decomp", syn["w"], syn["zn"], syn["zn_err"], discard=100, thin=2, rtd=True, model_curves=True, **kw)
ref = bb.BatchInversion("decomp", syn["w"], syn["zn"], syn["zn_err"], **kw).fit(discard=100, thin=2, rtd=True,
                                                                                model_curves=True)
for k in NEW_KEYS + ("percentiles", "mean", "std", "acceptance_fraction", "flags"):
    np.testing.assert_array_equal(res[k], ref[k])            # independent of the number of ranks
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_products_two_ranks_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker_products.py"
    script.write_text(_NCCL_WORKER)
    port = str(29690 + os.getpid() % 190)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out
        assert "ok" in out
