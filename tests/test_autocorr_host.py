"""Per-spectrum autocorrelation times in batch results, the parts that need no GPU: the result table's `<name>_tau`
columns, the empty-shard shape of `fit_device(autocorr=True)`, and the argument checks of `bisip_autocorr_time`."""
import ctypes as C

import numpy as np
import pytest


def _results(B=4, ndim=3, npct=3, tau=False):
    rng = np.random.default_rng(7)
    r = {'mean': rng.standard_normal((B, ndim)), 'std': rng.random((B, ndim)),
         'percentiles': rng.standard_normal((B, npct, ndim)), 'acceptance_fraction': rng.random(B),
         'flags': np.array([0, 1, 0, 2][:B], dtype=np.int32)}
    if tau:
        r['autocorr_time'] = 1 + 10 * rng.random((B, ndim))
    return r


def test_batch_table_without_autocorr_is_unchanged():
    from bisip_b200.products import batch_table
    names = ['r0', 'm', 'c']
    res = _results()
    cols, table = batch_table(names, res, ids=np.arange(10, 14), percentiles=(2.5, 50, 97.5))
    want_cols = (['spectrum', 'acceptance_fraction', 'flags'] + [f'{n}_mean' for n in names] + [f'{n}_std' for n in names]
                 + [f'{n}_p{q}' for q in ('2.5', '50', '97.5') for n in names])
    assert cols == want_cols
    want = np.concatenate([np.arange(10, 14, dtype=np.float64)[:, None], res['acceptance_fraction'][:, None],
                           res['flags'].astype(np.float64)[:, None], res['mean'], res['std'],
                           res['percentiles'][:, 0], res['percentiles'][:, 1], res['percentiles'][:, 2]], axis=1)
    np.testing.assert_array_equal(table, want)


def test_batch_table_appends_tau_columns_after_the_percentiles(tmp_path):
    from bisip_b200.products import batch_table
    names = ['r0', 'm', 'c']
    res = _results(tau=True)
    plain = {k: v for k, v in res.items() if k != 'autocorr_time'}
    cols0, table0 = batch_table(names, plain)
    cols, table = batch_table(names, res)
    assert cols == cols0 + ['r0_tau', 'm_tau', 'c_tau']
    np.testing.assert_array_equal(table[:, :len(cols0)], table0)
    np.testing.assert_array_equal(table[:, len(cols0):], res['autocorr_time'])


def test_empty_shard_fit_device_autocorr_shape(monkeypatch):
    import torch
    from bisip_b200 import _lib
    from bisip_b200.batch import BatchInversion
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))
    w = np.logspace(3, -1, 8)
    inv = BatchInversion('dias', w, np.zeros((0, 2, 8)), np.ones((0, 2, 8)), nwalkers=16, nsteps=10)
    out = inv.fit_device(discard=4, autocorr=True)
    assert out['autocorr_time'].shape == (0, 5) and out['autocorr_time'].dtype == torch.float64
    assert 'autocorr_time' not in inv.fit_device(discard=4)


def test_autocorr_time_argument_checks():
    """Every check runs before the library touches a device, so the documented codes are testable without one."""
    from bisip_b200 import _lib
    lib = _lib.load()
    out = (C.c_double * 4)()
    fake = C.c_void_p(0x1000)            # never dereferenced: the call returns before any launch
    args = dict(data=fake, B=2, n=10, W=8, ncol=2, c=5.0, out=C.cast(out, C.c_void_p))

    def call(**kw):
        a = dict(args, **kw)
        return lib.bisip_autocorr_time(a['data'], a['B'], a['n'], a['W'], a['ncol'], a['c'], a['out'], None)

    bad, unsupported = -1, -2
    assert call(data=C.c_void_p(0)) == bad
    assert call(out=C.c_void_p(0)) == bad
    for k in ('B', 'n', 'W', 'ncol'):
        assert call(**{k: 0}) == bad, k
        assert call(**{k: -3}) == bad, k
    for c in (0.0, -1.0, float('nan'), float('inf')):
        assert call(c=c) == bad, c
    assert 'c must be' in lib.bisip_last_error().decode()
    assert call(B=65536) == unsupported
    assert 'n_spectra' in lib.bisip_last_error().decode()
