"""RTD, total-chargeability and model-curve products of batch fits, the parts that need no GPU: the result table's
`total_m_*` columns, the empty-shard shapes of `fit_device(rtd=True, model_curves=True)`, the argument checks of
`bisip_rtd_stats`, and the gather of the new keys by a two-rank `fit_sharded`."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _results(B=4, ndim=3, npct=3, tau=False, total=False):
    rng = np.random.default_rng(11)
    r = {'mean': rng.standard_normal((B, ndim)), 'std': rng.random((B, ndim)),
         'percentiles': rng.standard_normal((B, npct, ndim)), 'acceptance_fraction': rng.random(B),
         'flags': np.array([0, 1, 0, 2][:B], dtype=np.int32)}
    if tau:
        r['autocorr_time'] = 1 + 10 * rng.random((B, ndim))
    if total:
        r['rtd_percentiles'] = rng.standard_normal((B, npct, 7))
        r['total_chargeability_percentiles'] = rng.standard_normal((B, npct))
        r['total_chargeability_mean'] = rng.standard_normal(B)
        r['total_chargeability_std'] = rng.random(B)
    return r


@pytest.mark.parametrize('tau', [False, True])
def test_batch_table_appends_total_m_columns_last(tau, tmp_path):
    from bisip_b200.products import batch_table
    names = ['r0', 'a0', 'a1']
    pct = (16, 50, 84)
    res = _results(tau=tau, total=True)
    plain = {k: v for k, v in res.items() if not k.startswith(('total_', 'rtd_'))}
    cols0, table0 = batch_table(names, plain, percentiles=pct)
    cols, table = batch_table(names, res, percentiles=pct)
    assert cols == cols0 + ['total_m_mean', 'total_m_std', 'total_m_p16', 'total_m_p50', 'total_m_p84']
    if tau:
        assert cols0[-3:] == ['r0_tau', 'a0_tau', 'a1_tau']
    np.testing.assert_array_equal(table[:, :len(cols0)], table0)
    np.testing.assert_array_equal(table[:, len(cols0)], res['total_chargeability_mean'])
    np.testing.assert_array_equal(table[:, len(cols0) + 1], res['total_chargeability_std'])
    np.testing.assert_array_equal(table[:, len(cols0) + 2:], res['total_chargeability_percentiles'])
    # without the total chargeability the table is the one of the parent layout, byte for byte in the CSV
    p0, p1 = tmp_path / 'a.csv', tmp_path / 'b.csv'
    for path, r in ((p0, plain), (p1, {k: v for k, v in res.items() if k.startswith('rtd_') or k in plain})):
        c, t = batch_table(names, r, percentiles=pct)
        np.savetxt(path, t, header=','.join(c), delimiter=',', comments='')
    assert p0.read_bytes() == p1.read_bytes()


def _cpu(monkeypatch):
    import torch
    from bisip_b200 import _lib
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))


def test_empty_shard_fit_device_product_shapes(monkeypatch):
    import torch
    from bisip_b200.batch import BatchInversion
    _cpu(monkeypatch)
    N = 8
    w = np.logspace(3, -1, N)
    inv = BatchInversion('decomp', w, np.zeros((0, 2, N)), np.ones((0, 2, N)), nwalkers=16, nsteps=10, poly_deg=3,
                         n_tau=20)
    out = inv.fit_device(discard=4, percentiles=(5, 50, 95, 99), rtd=True, model_curves=True)
    want = {'rtd_percentiles': (0, 4, 20), 'rtd_mean': (0, 20), 'rtd_std': (0, 20),
            'total_chargeability_percentiles': (0, 4), 'total_chargeability_mean': (0,),
            'total_chargeability_std': (0,), 'model_percentiles': (0, 4, 2, N)}
    for k, shape in want.items():
        assert tuple(out[k].shape) == shape, k
        assert out[k].dtype == torch.float64, k
    plain = inv.fit_device(discard=4)
    assert set(plain) == {'percentiles', 'mean', 'std', 'acceptance_fraction', 'flags'}
    assert set(inv.fit_device(discard=4, model_curves=True)) == set(plain) | {'model_percentiles'}
    # per-spectrum grids (w of shape (B, N)) on an empty shard
    per = BatchInversion('decomp', np.zeros((0, N)), np.zeros((0, 2, N)), np.ones((0, 2, N)), nwalkers=16, nsteps=10,
                         poly_deg=3, n_tau=20)
    assert tuple(per.fit_device(discard=4, rtd=True)['rtd_percentiles'].shape) == (0, 3, 20)
    # Cole-Cole model curves: 2 modes, ndim 7
    cc = BatchInversion('colecole', w, np.zeros((0, 2, N)), np.ones((0, 2, N)), nwalkers=16, nsteps=10, n_modes=2)
    assert tuple(cc.fit_device(discard=4, model_curves=True)['model_percentiles'].shape) == (0, 3, 2, N)


def test_rtd_on_other_models_raises_before_sampling(monkeypatch):
    from bisip_b200 import engine
    from bisip_b200.batch import BatchInversion
    _cpu(monkeypatch)

    def no_launch(*a, **k):
        raise AssertionError('sampled')
    monkeypatch.setattr(engine, 'ensemble_run', no_launch)
    w = np.logspace(3, -1, 8)
    for model in ('dias', 'shin', 'colecole'):
        inv = BatchInversion(model, w, np.zeros((2, 2, 8)), np.ones((2, 2, 8)), nwalkers=16, nsteps=10)
        with pytest.raises(ValueError, match='decomp'):
            inv.fit(discard=4, rtd=True)
        with pytest.raises(ValueError, match='decomp'):
            inv.fit_device(discard=4, rtd=True)


def test_rtd_stats_argument_checks():
    """Every check runs before the library touches a device, so the documented codes are testable without one."""
    from bisip_b200 import _lib
    lib = _lib.load()
    lo = (C.c_int64 * 17)(*([0] * 17))
    ga = (C.c_double * 17)(*([0.5] * 17))
    fake = C.c_void_p(0x1000)            # never dereferenced: the call returns before any launch
    args = dict(B=2, n=10, ndim=6, n_coef=5, n_tau=8, theta=fake, lt=fake, stride=0, npct=3, lo=lo, ga=ga, pct=fake,
                mean=fake, std=fake)

    def call(**kw):
        a = dict(args, **kw)
        return lib.bisip_rtd_stats(a['B'], a['n'], a['ndim'], a['n_coef'], a['n_tau'], a['theta'], a['lt'], a['stride'],
                                   a['npct'], a['lo'], a['ga'], a['pct'], a['mean'], a['std'], None)

    def err():
        return lib.bisip_last_error().decode()

    bad, unsupported, null = -1, -2, C.c_void_p(0)
    for k in ('theta', 'lt'):
        assert call(**{k: null}) == bad, k
        assert 'bad argument' in err()
    for k in ('B', 'n', 'ndim', 'n_coef', 'n_tau'):
        assert call(**{k: 0}) == bad, k
        assert call(**{k: -3}) == bad, k
        assert 'bad argument' in err()
    assert call(stride=-1) == bad and 'bad argument' in err()
    assert call(npct=-1) == bad and 'bad argument' in err()
    assert call(ndim=5) == bad and 'ndim != 1 + n_coef' in err()
    assert call(ndim=7) == bad and 'ndim != 1 + n_coef' in err()
    for k in ('lo', 'ga', 'pct'):
        assert call(**{k: None}) == bad, k
        assert 'percentile arrays null' in err()
    assert call(npct=0, pct=null, mean=null, std=null) == bad and 'no output' in err()
    assert call(npct=17) == unsupported and 'at most 16 percentiles' in err()
    assert call(B=65536) == unsupported and 'n_spectra > 65535' in err()
    assert call(n_coef=33, ndim=34) == unsupported and 'n_coef > 32' in err()


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
S, N = 7, 8
seen = []
def fake_fit_device(self, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), keep_chain=False, batch_size=None,
                    _chain_to_host=False, autocorr=False, rtd=False, model_curves=False):
    seen.append((autocorr, rtd, model_curves))
    B, P = self.n_spectra, len(percentiles)
    g = torch.arange(self.spectrum_offset, self.spectrum_offset + B, dtype=torch.float64)
    f = dict(dtype=torch.float64)
    out = {"percentiles": g[:, None, None] * torch.ones(1, P, self.ndim, **f), "mean": g[:, None] * torch.ones(1, self.ndim, **f),
           "std": g[:, None] * torch.ones(1, self.ndim, **f), "acceptance_fraction": 0.01 * g,
           "flags": torch.zeros(B, dtype=torch.int32)}
    if rtd:
        out["rtd_percentiles"] = g[:, None, None] + torch.arange(P * S, **f).reshape(1, P, S)
        out["rtd_mean"] = g[:, None] + torch.arange(S, **f)
        out["rtd_std"] = 2 * g[:, None] + torch.zeros(1, S, **f)
        out["total_chargeability_percentiles"] = g[:, None] + torch.arange(P, **f)
        out["total_chargeability_mean"] = 3 * g
        out["total_chargeability_std"] = 4 * g
    if model_curves:
        out["model_percentiles"] = g[:, None, None, None] + torch.arange(P * 2 * N, **f).reshape(1, P, 2, N)
    return out
batch.BatchInversion.fit_device = fake_fit_device
w = np.logspace(3, -1, N)
for B in (11, 1):                  # B = 1: rank 1 holds an empty shard and still takes part in the gather
    zn = np.zeros((B, 2, N)); ze = np.ones((B, 2, N))
    res = bisip_b200.fit_sharded("decomp", w, zn, ze, discard=2, percentiles=(5, 50, 95, 99), rtd=True,
                                 model_curves=True, nwalkers=12, nsteps=10, poly_deg=3, n_tau=S)
    g = np.arange(B, dtype=np.float64)
    assert res["rtd_percentiles"].shape == (B, 4, S) and res["rtd_mean"].shape == (B, S) and res["rtd_std"].shape == (B, S)
    assert res["total_chargeability_percentiles"].shape == (B, 4)
    assert res["total_chargeability_mean"].shape == (B,) and res["total_chargeability_std"].shape == (B,)
    assert res["model_percentiles"].shape == (B, 4, 2, N)
    np.testing.assert_array_equal(res["rtd_percentiles"][:, 3, 6], g + 27)
    np.testing.assert_array_equal(res["rtd_mean"][:, 2], g + 2)
    np.testing.assert_array_equal(res["total_chargeability_percentiles"][:, 1], g + 1)
    np.testing.assert_array_equal(res["total_chargeability_mean"], 3 * g)
    np.testing.assert_array_equal(res["total_chargeability_std"], 4 * g)
    np.testing.assert_array_equal(res["model_percentiles"][:, 2, 1, 5], g + 2 * 16 + 8 + 5)
    cols = res["inversion"].to_csv(os.path.join(os.environ["OUT"], f"r{rank}_{B}.csv"))
    assert cols[-6:] == ["total_m_mean", "total_m_std", "total_m_p5", "total_m_p50", "total_m_p95", "total_m_p99"]
plain = bisip_b200.fit_sharded("decomp", w, np.zeros((3, 2, N)), np.ones((3, 2, N)), discard=2, nwalkers=12, nsteps=10,
                               poly_deg=3, n_tau=S)
assert not any(k.startswith(("rtd_", "total_", "model_")) for k in plain)
assert seen == [(False, True, True), (False, True, True), (False, False, False)]
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_products_two_ranks_gloo(tmp_path):
    """The new keys go through the packed all-gather with the right shapes, also from a rank with an empty shard."""
    script = tmp_path / "worker_products.py"
    script.write_text(_SHARDED_WORKER)
    port = str(29700 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT, OUT=str(tmp_path))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert "ok" in out
