"""WAIC of batch fits, the parts that need no GPU: `products.compare_waic` against its NumPy definition, the result
table's WAIC columns, the empty-shard shapes and key sets of `fit_device(waic=True)`, the argument checks of
`bisip_waic`, and the gather of the WAIC keys by a two-rank `fit_sharded`."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WAIC_KEYS = {'elpd_waic', 'p_waic', 'se_elpd_waic', 'waic_pointwise', 'waic_n_high_p'}


def _waic_res(B, N, seed):
    rng = np.random.default_rng(seed)
    pw = rng.standard_normal((B, N)) - 3.0
    return {'elpd_waic': pw.sum(1), 'p_waic': rng.random(B), 'se_elpd_waic': rng.random(B), 'waic_pointwise': pw,
            'waic_n_high_p': rng.integers(0, N, B).astype(np.int32)}


def test_compare_waic_matches_numpy():
    from bisip_b200.products import compare_waic
    a, b = _waic_res(5, 12, 1), _waic_res(5, 12, 2)
    out = compare_waic(a, b)
    np.testing.assert_array_equal(out['elpd_diff'], a['elpd_waic'] - b['elpd_waic'])
    d = a['waic_pointwise'] - b['waic_pointwise']
    se = np.array([np.sqrt(12 * np.sum((r - r.mean()) ** 2) / 11) for r in d])
    np.testing.assert_allclose(out['se_diff'], se, rtol=1e-13)
    assert out['elpd_diff'].shape == (5,) and out['se_diff'].shape == (5,)
    same = compare_waic(a, a)
    np.testing.assert_array_equal(same['elpd_diff'], 0.0)
    np.testing.assert_array_equal(same['se_diff'], 0.0)
    # single-spectrum dicts (Inversion.get_waic): scalars
    one = compare_waic({'elpd_waic': 1.5, 'waic_pointwise': np.array([0.5, 1.0])},
                       {'elpd_waic': 0.5, 'waic_pointwise': np.array([0.0, 0.5])})
    assert float(one['elpd_diff']) == 1.0 and float(one['se_diff']) == 0.0


def test_compare_waic_shape_errors():
    from bisip_b200.products import compare_waic
    a = _waic_res(4, 10, 3)
    with pytest.raises(ValueError, match='shapes differ'):
        compare_waic(a, _waic_res(3, 10, 4))                  # other spectra
    with pytest.raises(ValueError, match='shapes differ'):
        compare_waic(a, _waic_res(4, 11, 4))                  # other frequencies
    bad = dict(a, waic_pointwise=a['waic_pointwise'][:3])
    with pytest.raises(ValueError, match='shapes differ'):
        compare_waic(bad, bad)                                # pointwise rows do not match elpd_waic


def test_batch_table_appends_waic_columns_last(tmp_path):
    from bisip_b200.products import batch_table
    rng = np.random.default_rng(7)
    B, ndim, names, pct = 4, 3, ['r0', 'a0', 'a1'], (16, 50, 84)
    plain = {'mean': rng.standard_normal((B, ndim)), 'std': rng.random((B, ndim)),
             'percentiles': rng.standard_normal((B, 3, ndim)), 'acceptance_fraction': rng.random(B),
             'flags': np.array([0, 1, 0, 2], dtype=np.int32), 'autocorr_time': rng.random((B, ndim)),
             'total_chargeability_mean': rng.random(B), 'total_chargeability_std': rng.random(B),
             'total_chargeability_percentiles': rng.random((B, 3))}
    res = dict(plain, **_waic_res(B, 9, 8))
    cols0, table0 = batch_table(names, plain, percentiles=pct)
    cols, table = batch_table(names, res, percentiles=pct)
    assert cols == cols0 + ['elpd_waic', 'p_waic', 'se_elpd_waic', 'waic_n_high_p']
    np.testing.assert_array_equal(table[:, :len(cols0)], table0)
    np.testing.assert_array_equal(table[:, len(cols0)], res['elpd_waic'])
    np.testing.assert_array_equal(table[:, len(cols0) + 1], res['p_waic'])
    np.testing.assert_array_equal(table[:, len(cols0) + 2], res['se_elpd_waic'])
    np.testing.assert_array_equal(table[:, len(cols0) + 3], res['waic_n_high_p'])
    # without the WAIC keys the CSV is byte-identical to the one written before they existed
    p0, p1 = tmp_path / 'a.csv', tmp_path / 'b.csv'
    for path, r in ((p0, plain), (p1, dict(plain, waic_pointwise=res['waic_pointwise']))):
        c, t = batch_table(names, r, percentiles=pct)
        np.savetxt(path, t, header=','.join(c), delimiter=',', comments='')
    assert p0.read_bytes() == p1.read_bytes()


def _cpu(monkeypatch):
    import torch
    from bisip_b200 import _lib
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))


@pytest.mark.parametrize('model,kw', [('decomp', dict(poly_deg=3, n_tau=20)), ('colecole', dict(n_modes=2)),
                                      ('dias', {}), ('shin', {})])
def test_empty_shard_fit_device_waic_shapes(monkeypatch, model, kw):
    import torch
    from bisip_b200.batch import BatchInversion
    _cpu(monkeypatch)
    N = 8
    inv = BatchInversion(model, np.logspace(3, -1, N), np.zeros((0, 2, N)), np.ones((0, 2, N)), nwalkers=16,
                         nsteps=10, **kw)
    out = inv.fit_device(discard=4, waic=True)
    want = {'elpd_waic': (0,), 'p_waic': (0,), 'se_elpd_waic': (0,), 'waic_pointwise': (0, N), 'waic_n_high_p': (0,)}
    for k, shape in want.items():
        assert tuple(out[k].shape) == shape, k
        assert out[k].dtype == (torch.int32 if k == 'waic_n_high_p' else torch.float64), k
    plain = inv.fit_device(discard=4)
    assert set(plain) == {'percentiles', 'mean', 'std', 'acceptance_fraction', 'flags'}
    assert set(out) == set(plain) | WAIC_KEYS
    assert set(inv.fit_device(discard=4, autocorr=True, waic=True)) == set(plain) | WAIC_KEYS | {'autocorr_time'}


def test_waic_argument_checks():
    """Every check runs before the library touches a device, so the documented codes are testable without one."""
    from bisip_b200 import _lib
    lib = _lib.load()
    fake = C.c_void_p(0x1000)            # never dereferenced: the call returns before any launch
    null = C.c_void_p(0)
    N = 8

    def desc(model=_lib.MODEL_DECOMP, ndim=6, n_modes=1, n_tau=20, n_coef=5, n_freq=N):
        return _lib.ModelDesc(model, ndim, n_freq, n_modes, n_tau, n_coef, _lib.PREC_FP64, 0, 1.0)

    ptrs = ('theta', 'w', 'taus', 'lt', 'y', 'yerr', 'lppd', 'p', 'elpd', 'pw', 'se', 'nh')
    args = dict(d=desc(), B=2, n=10, w_stride=0, tau_stride=0, **{k: fake for k in ptrs})

    def call(**kw):
        a = dict(args, **kw)
        d = a['d']
        return lib.bisip_waic(None if d is None else C.byref(d), a['B'], a['n'], a['theta'], a['w'], a['w_stride'],
                              a['taus'], a['lt'], a['tau_stride'], a['y'], a['yerr'], a['lppd'], a['p'], a['elpd'],
                              a['pw'], a['se'], a['nh'], None)

    def err():
        return lib.bisip_last_error().decode()

    bad, unsupported = -1, -2
    assert call(d=None) == bad and 'desc is null' in err()
    for k in ptrs:
        assert call(**{k: null}) == bad, k
        assert 'bisip_waic' in err() and ('bad argument' in err() or 'null' in err()), k
    for k in ('B', 'n'):
        assert call(**{k: 0}) == bad, k
        assert call(**{k: -3}) == bad, k
        assert 'bad argument' in err()
    assert call(n=1) == bad and 'bad argument' in err()           # the variance over samples needs two
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
                    _chain_to_host=False, waic=False):
    seen.append(waic)
    B, P = self.n_spectra, len(percentiles)
    g = torch.arange(self.spectrum_offset, self.spectrum_offset + B, dtype=torch.float64)
    f = dict(dtype=torch.float64)
    out = {"percentiles": g[:, None, None] * torch.ones(1, P, self.ndim, **f), "mean": g[:, None] * torch.ones(1, self.ndim, **f),
           "std": g[:, None] * torch.ones(1, self.ndim, **f), "acceptance_fraction": 0.01 * g,
           "flags": torch.zeros(B, dtype=torch.int32)}
    if waic:
        out["elpd_waic"] = -g
        out["p_waic"] = 0.5 * g
        out["se_elpd_waic"] = 0.25 * g
        out["waic_pointwise"] = g[:, None] + torch.arange(N, **f)
        out["waic_n_high_p"] = (g % 3).to(torch.int32)
    return out
batch.BatchInversion.fit_device = fake_fit_device
w = np.logspace(3, -1, N)
for B in (11, 1):                  # B = 1: rank 1 holds an empty shard and still takes part in the gather
    res = bisip_b200.fit_sharded("decomp", w, np.zeros((B, 2, N)), np.ones((B, 2, N)), discard=2, waic=True,
                                 nwalkers=12, nsteps=10, poly_deg=3, n_tau=7)
    g = np.arange(B, dtype=np.float64)
    np.testing.assert_array_equal(res["elpd_waic"], -g)
    np.testing.assert_array_equal(res["p_waic"], 0.5 * g)
    np.testing.assert_array_equal(res["se_elpd_waic"], 0.25 * g)
    assert res["waic_pointwise"].shape == (B, N)
    np.testing.assert_array_equal(res["waic_pointwise"][:, 5], g + 5)
    assert res["waic_n_high_p"].dtype == np.int32
    np.testing.assert_array_equal(res["waic_n_high_p"], (g % 3).astype(np.int32))
    cols = res["inversion"].to_csv(os.path.join(os.environ["OUT"], f"r{rank}_{B}.csv"))
    assert cols[-4:] == ["elpd_waic", "p_waic", "se_elpd_waic", "waic_n_high_p"]
plain = bisip_b200.fit_sharded("decomp", w, np.zeros((3, 2, N)), np.ones((3, 2, N)), discard=2, nwalkers=12, nsteps=10,
                               poly_deg=3, n_tau=7)
assert not any("waic" in k for k in plain)
assert seen == [True, True, False]
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_waic_two_ranks_gloo(tmp_path):
    """The WAIC keys go through the packed all-gather with their shapes and dtypes, also from an empty shard; without
    ``waic`` the keyword is not passed to ``fit_device`` at all."""
    script = tmp_path / "worker_waic.py"
    script.write_text(_SHARDED_WORKER)
    port = str(29800 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT, OUT=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert "ok" in out
