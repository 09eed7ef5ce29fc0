"""PSIS-LOO of batch fits, the parts that need no GPU: the NumPy restatement of the definition (`_ref_psis_loo`, which
the GPU parity tests compare against) checked on its own, `products.compare_loo` against its NumPy definition, the
result table's LOO columns, the empty-shard shapes and key sets of `fit_device(loo=True)`, the argument checks of
`bisip_psis_loo`, and the gather of the LOO keys by a two-rank `fit_sharded`."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.special import logsumexp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOO_KEYS = {'elpd_loo', 'p_loo', 'se_elpd_loo', 'loo_pointwise', 'pareto_k', 'loo_n_high_k'}
EPS = np.finfo(float).eps


def _gpdfit(u):
    """Zhang & Stephens generalized Pareto fit of the ascending u, with the weakly informative prior on k: (k, sigma)."""
    n = len(u)
    m = 30 + int(np.sqrt(n))
    b = 1 - np.sqrt(m / (np.arange(1, m + 1, dtype=float) - 0.5))
    b /= 3 * u[int(n / 4 + 0.5) - 1]
    b += 1 / u[-1]
    k = np.log1p(-b[:, None] * u).mean(axis=1)
    ls = n * (np.log(-(b / k)) - k - 1)
    with np.errstate(over='ignore'):
        w = 1 / np.exp(ls - ls[:, None]).sum(axis=1)          # an overflow gives w = 0
    keep = w >= 10 * EPS
    w = w[keep] / w[keep].sum()
    bp = np.sum(b[keep] * w)
    kh = np.log1p(-bp * u).mean()
    return (n * kh + 5) / (n + 10), -kh / bp


def _gpinv(p, k, sigma):
    if sigma <= 0:
        return np.full_like(p, np.nan)
    if abs(k) < EPS:
        return -np.log1p(-p) * sigma
    return np.expm1(-k * np.log1p(-p)) / k * sigma


def _ref_psis_loo(ll):
    """The definition, in NumPy, for one spectrum: ll (S, N) pointwise log-likelihood.  Besides the outputs it returns
    per frequency the relative gap between the M-th and (M+1)-th largest log-ratio (how unambiguous the tail set is)
    and whether the truncation at 0 changed a smoothed value."""
    S, N = ll.shape
    M = int(np.ceil(min(0.2 * S, 3 * np.sqrt(S))))
    elpd, p, k = np.empty(N), np.empty(N), np.empty(N)
    gap, truncated = np.empty(N), np.zeros(N, dtype=bool)
    for j in range(N):
        lj = ll[:, j]
        lppd = logsumexp(lj) - np.log(S)
        x = -lj - np.max(-lj)
        xs = np.sort(x)
        cutoff = max(xs[-M - 1], np.log(np.finfo(float).tiny))
        gap[j] = (xs[-M] - xs[-M - 1]) / max(1.0, abs(xs[-M - 1]))
        tail = np.flatnonzero(x > cutoff)
        L = len(tail)
        xt = x.copy()
        if L <= 4:
            k[j] = np.inf
        else:
            order = tail[np.argsort(x[tail], kind='stable')]
            k[j], sigma = _gpdfit(np.exp(x[order]) - np.exp(cutoff))
            if np.isfinite(k[j]):
                sm = np.log(_gpinv((np.arange(L) + 0.5) / L, k[j], sigma) + np.exp(cutoff))
                truncated[j] = bool(np.any(sm > 0))
                xt[order] = sm
                xt = np.minimum(xt, 0)
        elpd[j] = logsumexp(xt + lj) - logsumexp(xt)
        p[j] = lppd - elpd[j]
    thr = min(1 - 1 / np.log10(S), 0.7)
    out = dict(elpd_i=elpd, p_i=p, pareto_k=k, elpd=elpd.sum(), p_loo=p.sum(), se=np.sqrt(N * np.var(elpd, ddof=1)),
               n_high_k=int(np.count_nonzero(k > thr)), threshold=thr, gap=gap, truncated=truncated)
    if np.isnan(ll).any():
        for key in ('elpd_i', 'p_i', 'pareto_k'):
            out[key] = np.full(N, np.nan)
        out.update(elpd=np.nan, p_loo=np.nan, se=np.nan, n_high_k=0)
    return out


@pytest.mark.parametrize('c', [-0.2, 0.3, 0.8])
def test_ref_gpdfit_recovers_genpareto_shape(c):
    from scipy.stats import genpareto
    u = np.sort(genpareto.rvs(c, scale=1.5, size=2000, random_state=np.random.default_rng(2026)))
    k, sigma = _gpdfit(u)
    assert abs(k - c) < 0.05, (k, c)
    assert sigma > 0


def test_ref_short_tail_is_plain_importance_sampling():
    """S = 20: M = 4, so the tail never has more than 4 samples: k = inf and no smoothing, which leaves the raw
    importance-sampling estimate -(logsumexp(-ll) - ln S)."""
    ll = np.random.default_rng(3).normal(-2.0, 1.5, (20, 7))
    r = _ref_psis_loo(ll)
    assert np.all(np.isinf(r['pareto_k'])) and r['n_high_k'] == 7
    np.testing.assert_allclose(r['elpd_i'], -(logsumexp(-ll, axis=0) - np.log(20)), rtol=1e-14, atol=1e-14)


def test_ref_invariant_to_a_constant_shift():
    """ll + c leaves the importance ratios, so k and elpd_loo_j - lppd_j, unchanged."""
    ll = np.random.default_rng(5).normal(0.0, np.array([0.5, 1.5, 3.0, 1.0]), (4000, 4))
    a, b = _ref_psis_loo(ll), _ref_psis_loo(ll + 37.25)
    assert np.all(np.isfinite(a['pareto_k']))
    np.testing.assert_allclose(b['pareto_k'], a['pareto_k'], rtol=0, atol=1e-9)
    np.testing.assert_allclose(b['p_i'], a['p_i'], rtol=0, atol=1e-9)      # p_i = lppd - elpd_loo
    np.testing.assert_allclose(b['elpd_i'] - a['elpd_i'], 37.25, rtol=0, atol=1e-9)


def _loo_res(B, N, seed):
    rng = np.random.default_rng(seed)
    pw = rng.standard_normal((B, N)) - 3.0
    return {'elpd_loo': pw.sum(1), 'p_loo': rng.random(B), 'se_elpd_loo': rng.random(B), 'loo_pointwise': pw,
            'pareto_k': rng.random((B, N)), 'loo_n_high_k': rng.integers(0, N, B).astype(np.int32)}


def test_compare_loo_matches_numpy():
    from bisip_b200.products import compare_loo
    a, b = _loo_res(5, 12, 1), _loo_res(5, 12, 2)
    out = compare_loo(a, b)
    np.testing.assert_array_equal(out['elpd_diff'], a['elpd_loo'] - b['elpd_loo'])
    d = a['loo_pointwise'] - b['loo_pointwise']
    se = np.array([np.sqrt(12 * np.sum((r - r.mean()) ** 2) / 11) for r in d])
    np.testing.assert_allclose(out['se_diff'], se, rtol=1e-13)
    assert out['elpd_diff'].shape == (5,) and out['se_diff'].shape == (5,)
    same = compare_loo(a, a)
    np.testing.assert_array_equal(same['elpd_diff'], 0.0)
    np.testing.assert_array_equal(same['se_diff'], 0.0)
    # single-spectrum dicts (Inversion.get_loo): scalars
    one = compare_loo({'elpd_loo': 1.5, 'loo_pointwise': np.array([0.5, 1.0])},
                      {'elpd_loo': 0.5, 'loo_pointwise': np.array([0.0, 0.5])})
    assert float(one['elpd_diff']) == 1.0 and float(one['se_diff']) == 0.0


def test_compare_loo_shape_errors():
    from bisip_b200.products import compare_loo
    a = _loo_res(4, 10, 3)
    with pytest.raises(ValueError, match='compare_loo: shapes differ'):
        compare_loo(a, _loo_res(3, 10, 4))                    # other spectra
    with pytest.raises(ValueError, match='compare_loo: shapes differ'):
        compare_loo(a, _loo_res(4, 11, 4))                    # other frequencies
    bad = dict(a, loo_pointwise=a['loo_pointwise'][:3])
    with pytest.raises(ValueError, match='loo_pointwise'):
        compare_loo(bad, bad)                                 # pointwise rows do not match elpd_loo


def test_batch_table_appends_loo_columns_last(tmp_path):
    from bisip_b200.products import batch_table
    rng = np.random.default_rng(7)
    B, ndim, names, pct = 4, 3, ['r0', 'a0', 'a1'], (16, 50, 84)
    plain = {'mean': rng.standard_normal((B, ndim)), 'std': rng.random((B, ndim)),
             'percentiles': rng.standard_normal((B, 3, ndim)), 'acceptance_fraction': rng.random(B),
             'flags': np.array([0, 1, 0, 2], dtype=np.int32), 'autocorr_time': rng.random((B, ndim)),
             'elpd_waic': rng.random(B), 'p_waic': rng.random(B), 'se_elpd_waic': rng.random(B),
             'waic_pointwise': rng.random((B, 9)), 'waic_n_high_p': np.arange(B, dtype=np.int32)}
    res = dict(plain, **_loo_res(B, 9, 8))
    cols0, table0 = batch_table(names, plain, percentiles=pct)
    cols, table = batch_table(names, res, percentiles=pct)
    assert cols0[-4:] == ['elpd_waic', 'p_waic', 'se_elpd_waic', 'waic_n_high_p']
    assert cols == cols0 + ['elpd_loo', 'p_loo', 'se_elpd_loo', 'loo_n_high_k']
    np.testing.assert_array_equal(table[:, :len(cols0)], table0)
    for i, k in enumerate(('elpd_loo', 'p_loo', 'se_elpd_loo', 'loo_n_high_k')):
        np.testing.assert_array_equal(table[:, len(cols0) + i], res[k])
    # without the LOO totals the CSV is byte-identical to the one written before they existed
    p0, p1 = tmp_path / 'a.csv', tmp_path / 'b.csv'
    for path, r in ((p0, plain), (p1, dict(plain, loo_pointwise=res['loo_pointwise'], pareto_k=res['pareto_k']))):
        c, t = batch_table(names, r, percentiles=pct)
        np.savetxt(path, t, header=','.join(c), delimiter=',', comments='')
    assert p0.read_bytes() == p1.read_bytes()


def _cpu(monkeypatch):
    import torch
    from bisip_b200 import _lib
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))


@pytest.mark.parametrize('model,kw', [('decomp', dict(poly_deg=3, n_tau=20)), ('colecole', dict(n_modes=2)),
                                      ('dias', {}), ('shin', {})])
def test_empty_shard_fit_device_loo_shapes(monkeypatch, model, kw):
    import torch
    from bisip_b200.batch import BatchInversion
    _cpu(monkeypatch)
    N = 8
    inv = BatchInversion(model, np.logspace(3, -1, N), np.zeros((0, 2, N)), np.ones((0, 2, N)), nwalkers=16,
                         nsteps=10, **kw)
    out = inv.fit_device(discard=4, loo=True)
    want = {'elpd_loo': (0,), 'p_loo': (0,), 'se_elpd_loo': (0,), 'loo_pointwise': (0, N), 'pareto_k': (0, N),
            'loo_n_high_k': (0,)}
    for k, shape in want.items():
        assert tuple(out[k].shape) == shape, k
        assert out[k].dtype == (torch.int32 if k == 'loo_n_high_k' else torch.float64), k
    plain = inv.fit_device(discard=4)
    assert set(plain) == {'percentiles', 'mean', 'std', 'acceptance_fraction', 'flags'}
    assert set(out) == set(plain) | LOO_KEYS
    waic = set(inv.fit_device(discard=4, waic=True))
    assert set(inv.fit_device(discard=4, waic=True, loo=True)) == waic | LOO_KEYS
    assert set(inv.fit_device(discard=4, autocorr=True, loo=True)) == set(plain) | LOO_KEYS | {'autocorr_time'}


def test_psis_loo_argument_checks():
    """Every check runs before the library touches a device, so the documented codes are testable without one."""
    from bisip_b200 import _lib
    lib = _lib.load()
    fake = C.c_void_p(0x1000)            # never dereferenced: the call returns before any launch
    null = C.c_void_p(0)
    N = 8

    def desc(model=_lib.MODEL_DECOMP, ndim=6, n_modes=1, n_tau=20, n_coef=5, n_freq=N):
        return _lib.ModelDesc(model, ndim, n_freq, n_modes, n_tau, n_coef, _lib.PREC_FP64, 0, 1.0)

    ptrs = ('theta', 'w', 'taus', 'lt', 'y', 'yerr', 'elpd_i', 'p_i', 'k', 'elpd', 'p_loo', 'se', 'nh')
    args = dict(d=desc(), B=2, n=10, w_stride=0, tau_stride=0, **{k: fake for k in ptrs})

    def call(**kw):
        a = dict(args, **kw)
        d = a['d']
        return lib.bisip_psis_loo(None if d is None else C.byref(d), a['B'], a['n'], a['theta'], a['w'],
                                  a['w_stride'], a['taus'], a['lt'], a['tau_stride'], a['y'], a['yerr'], a['elpd_i'],
                                  a['p_i'], a['k'], a['elpd'], a['p_loo'], a['se'], a['nh'], None)

    def err():
        return lib.bisip_last_error().decode()

    bad, unsupported = -1, -2
    assert call(d=None) == bad and 'desc is null' in err()
    for k in ptrs:
        assert call(**{k: null}) == bad, k
        assert 'bisip_psis_loo' in err() and ('bad argument' in err() or 'null' in err()), k
    for k in ('B', 'n'):
        assert call(**{k: 0}) == bad, k
        assert call(**{k: -3}) == bad, k
        assert 'bad argument' in err()
    assert call(n=1) == bad and 'bad argument' in err()           # leave-one-out needs two samples
    assert call(tau_stride=-1) == bad and 'bad argument' in err()
    assert call(w_stride=-1) == bad and 'bad argument' in err()
    assert call(d=desc(n_freq=0)) == bad
    assert call(d=desc(ndim=5)) == bad and 'n_coef' in err()
    assert call(d=desc(n_coef=0, ndim=1)) == bad
    assert call(d=desc(n_tau=0)) == bad
    assert call(d=desc(model=_lib.MODEL_COLECOLE, ndim=6, n_modes=2)) == bad and 'ndim' in err()
    assert call(d=desc(model=_lib.MODEL_DIAS, ndim=6)) == bad and 'ndim' in err()
    assert call(d=desc(model=_lib.MODEL_SHIN, ndim=5)) == bad and 'ndim' in err()
    assert call(d=desc(model=7)) == bad and 'unknown model' in err()
    assert call(B=65536) == unsupported and 'n_spectra > 65535' in err()
    assert call(d=desc(n_coef=33, ndim=34)) == unsupported and 'n_coef' in err()


_SHARDED_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"])
import numpy as np, torch, torch.distributed as dist
import bisip_b200
from bisip_b200 import _lib, batch
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
# the device work is stubbed: per-spectrum results are functions of the GLOBAL spectrum index, on CPU tensors
_lib.require_cuda = lambda device=None: torch.device("cpu")
N = 8
seen = []
def fake_fit_device(self, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), keep_chain=False, batch_size=None,
                    _chain_to_host=False, loo=False):
    seen.append(loo)
    B, P = self.n_spectra, len(percentiles)
    g = torch.arange(self.spectrum_offset, self.spectrum_offset + B, dtype=torch.float64)
    f = dict(dtype=torch.float64)
    out = {"percentiles": g[:, None, None] * torch.ones(1, P, self.ndim, **f), "mean": g[:, None] * torch.ones(1, self.ndim, **f),
           "std": g[:, None] * torch.ones(1, self.ndim, **f), "acceptance_fraction": 0.01 * g,
           "flags": torch.zeros(B, dtype=torch.int32)}
    if loo:
        out["elpd_loo"] = -g
        out["p_loo"] = 0.5 * g
        out["se_elpd_loo"] = 0.25 * g
        out["loo_pointwise"] = g[:, None] + torch.arange(N, **f)
        out["pareto_k"] = 0.1 * g[:, None] - torch.arange(N, **f)
        out["loo_n_high_k"] = (g % 3).to(torch.int32)
    return out
batch.BatchInversion.fit_device = fake_fit_device
w = np.logspace(3, -1, N)
for B in (11, 1):                  # B = 1: rank 1 holds an empty shard and still takes part in the gather
    res = bisip_b200.fit_sharded("decomp", w, np.zeros((B, 2, N)), np.ones((B, 2, N)), discard=2, loo=True,
                                 nwalkers=12, nsteps=10, poly_deg=3, n_tau=7)
    g = np.arange(B, dtype=np.float64)
    np.testing.assert_array_equal(res["elpd_loo"], -g)
    np.testing.assert_array_equal(res["p_loo"], 0.5 * g)
    np.testing.assert_array_equal(res["se_elpd_loo"], 0.25 * g)
    assert res["loo_pointwise"].shape == (B, N) and res["pareto_k"].shape == (B, N)
    np.testing.assert_array_equal(res["loo_pointwise"][:, 5], g + 5)
    np.testing.assert_array_equal(res["pareto_k"][:, 3], 0.1 * g - 3)
    assert res["loo_n_high_k"].dtype == np.int32
    np.testing.assert_array_equal(res["loo_n_high_k"], (g % 3).astype(np.int32))
    cols = res["inversion"].to_csv(os.path.join(os.environ["OUT"], f"r{rank}_{B}.csv"))
    assert cols[-4:] == ["elpd_loo", "p_loo", "se_elpd_loo", "loo_n_high_k"]
plain = bisip_b200.fit_sharded("decomp", w, np.zeros((3, 2, N)), np.ones((3, 2, N)), discard=2, nwalkers=12, nsteps=10,
                               poly_deg=3, n_tau=7)
assert not any("loo" in k or "pareto" in k for k in plain)
assert seen == [True, True, False]
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_loo_two_ranks_gloo(tmp_path):
    """The LOO keys go through the packed all-gather with their shapes and dtypes, also from an empty shard; without
    ``loo`` the keyword is not passed to ``fit_device`` at all."""
    script = tmp_path / "worker_loo.py"
    script.write_text(_SHARDED_WORKER)
    port = str(29400 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT, OUT=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert "ok" in out
