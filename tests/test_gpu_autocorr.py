"""Per-spectrum integrated autocorrelation times on the GPU (`bisip_autocorr_time`, `fit(..., autocorr=True)`):
parity with emcee's estimator on synthetic AR(1) chains and on fitted chains, NaN semantics, independence from batch
composition / sub-batching / sharding, and one launch per sub-batch."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHIS = (0.5, 0.8, 0.95)       # AR(1): tau = (1 + phi) / (1 - phi) = 3, 9, 39


def _ar1(B, n, W, ncol, seed):
    """(B, n, W, ncol) AR(1) chains, stationary start, offset from 0 so that the centring matters."""
    rng = np.random.default_rng(seed)
    phi = np.array(PHIS)[(np.arange(B)[:, None] + np.arange(ncol)[None, :]) % 3][:, None, :]     # (B, 1, ncol)
    e = rng.standard_normal((B, n, W, ncol))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1 - phi ** 2)
    for t in range(1, n):
        x[:, t] = phi * x[:, t - 1] + e[:, t]
    return x + 3.0


def _last_lag_window(x, c=5.0):
    """(ncol,) True where emcee's window of the column (n_t, n_w, n_d) is its last lag.  tau there is 0 in exact
    arithmetic, so every implementation returns rounding noise around 0: those columns are compared with atol."""
    from bisip_b200 import sampler
    n_t, n_w, n_d = x.shape
    out = np.zeros(n_d, dtype=bool)
    for d in range(n_d):
        f = sum(sampler.function_1d(x[:, k, d]) for k in range(n_w)) / n_w
        out[d] = sampler._auto_window(2.0 * np.cumsum(f) - 1.0, c) == n_t - 1
    return out


def _assert_tau_close(got, ref, last, rtol):
    np.testing.assert_allclose(got[~last], ref[~last], rtol=rtol, atol=0)
    np.testing.assert_allclose(got[last], ref[last], rtol=0, atol=1e-12)      # noise around 0 (see _last_lag_window)


def _dev(a):
    from bisip_b200 import _lib
    return _lib.dev_f64(a, _lib.require_cuda())


@pytest.mark.parametrize('B,n,W,ncol', [
    (3, 50, 2, 1), (3, 600, 32, 6), (2, 50, 33, 13), (3, 50, 256, 6), (2, 600, 300, 1), (2, 2, 256, 6),
    (1, 3000, 32, 2),            # 768 KB column: past one CTA's shared memory, the global-memory path
])
def test_autocorr_time_matches_emcee_on_ar1_chains(B, n, W, ncol):
    from bisip_b200 import engine, sampler
    x = _ar1(B, n, W, ncol, seed=B * 1000 + n + W + ncol)
    xd = _dev(x)
    got = engine.autocorr_time(xd).cpu().numpy()
    assert got.shape == (B, ncol)
    batch = sampler.integrated_time_batch(xd, c=5).cpu().numpy()
    for b in range(B):
        last = _last_lag_window(x[b])
        _assert_tau_close(got[b], sampler.integrated_time(x[b], c=5, quiet=True), last, rtol=1e-9)
        _assert_tau_close(got[b], batch[b], last, rtol=1e-10)
    # a spectrum's result depends on its own column only
    np.testing.assert_array_equal(engine.autocorr_time(_dev(x[B - 1:])).cpu().numpy(), got[B - 1:])
    if n >= 600:                         # and it estimates the AR(1) value (emcee's window biases it low on short chains)
        phi = np.array(PHIS)[np.arange(B) % 3]
        true = (1 + phi) / (1 - phi)
        assert np.all(np.abs(got[:, 0] - true) < 0.5 * true)


def test_autocorr_time_nan_semantics():
    from bisip_b200 import engine, sampler
    x = _ar1(2, 40, 8, 3, seed=5)
    x[0, :, 3, 1] = 2.5                  # a constant walker: 0/0 in its normalised ACF
    x[1, 17, 5, 2] = np.nan              # one NaN sample
    got = engine.autocorr_time(_dev(x)).cpu().numpy()
    np.testing.assert_array_equal(np.isnan(got), [[False, True, False], [False, False, True]])
    with np.errstate(invalid='ignore', divide='ignore'):
        for b in range(2):
            ref = sampler.integrated_time(x[b], quiet=True)
            np.testing.assert_array_equal(np.isnan(ref), np.isnan(got[b]))
            ok = ~np.isnan(ref)
            np.testing.assert_allclose(got[b][ok], ref[ok], rtol=1e-9)
    assert np.all(np.isnan(engine.autocorr_time(_dev(x[:, :1])).cpu().numpy()))       # n_keep == 1


def _survey(model, B, N=16, **kw):
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion
    _, w = synthetic.frequencies(N)
    probe = BatchInversion(model, w, np.zeros((1, 2, N)), np.ones((1, 2, N)), **kw)
    fwd = lambda th, ww: engine.forward(probe._spec(), _lib.dev_f64(th[:, None, :], probe.device),
                                        _lib.dev_f64(ww, probe.device))[:, 0].cpu().numpy()
    extra = {k: kw[k] for k in ('poly_deg', 'n_tau') if k in kw}
    return synthetic.make(model, 0, B, fwd, N=N, **extra)


FIT_CASES = {
    'decomp-fp64': ('decomp', dict(poly_deg=4, n_tau=32)),
    'decomp-fp64-collapsed': ('decomp', dict(poly_deg=4, n_tau=32, precision='fp64-collapsed')),
    'dias': ('dias', {}),
}


@pytest.mark.parametrize('case', sorted(FIT_CASES))
def test_fit_autocorr_time(case):
    import bisip_b200 as bb
    from bisip_b200 import _lib, sampler
    model, kw = FIT_CASES[case]
    B, discard, thin = 6, 200, 2
    syn = _survey(model, B, **kw)
    ctor = dict(nwalkers=32, nsteps=600, seed=17, **kw)
    inv = bb.BatchInversion(model, syn['w'], syn['zn'], syn['zn_err'], **ctor)
    full = inv.fit(discard=discard, thin=thin, keep_chain=True, autocorr=True)
    tau = full['autocorr_time']
    assert tau.shape == (B, inv.ndim) and np.all(np.isfinite(tau))
    for b in range(B):
        _assert_tau_close(tau[b], thin * sampler.integrated_time(full['chain'][b], quiet=True),
                          _last_lag_window(full['chain'][b]), rtol=1e-9)
    np.testing.assert_array_equal(inv.get_autocorr_time(thin=thin), tau)
    plain = inv.fit(discard=discard, thin=thin, keep_chain=True)
    assert 'autocorr_time' not in plain
    for k in plain:
        np.testing.assert_array_equal(full[k], plain[k], err_msg=k)
    np.testing.assert_array_equal(inv.fit(discard=discard, thin=thin, autocorr=True)['autocorr_time'], tau)
    n0 = _lib.launch_count()
    inv.fit(discard=discard, thin=thin, batch_size=3)
    n1 = _lib.launch_count()
    sub = inv.fit(discard=discard, thin=thin, batch_size=3, autocorr=True)
    n2 = _lib.launch_count()
    assert (n2 - n1) - (n1 - n0) == 2                     # one launch per sub-batch
    np.testing.assert_array_equal(sub['autocorr_time'], tau)
    np.testing.assert_array_equal(inv.fit_gathered(B, discard=discard, thin=thin, autocorr=True)['autocorr_time'], tau)
    sh = bb.fit_sharded(model, syn['w'], syn['zn'], syn['zn_err'], discard=discard, thin=thin, autocorr=True, **ctor)
    np.testing.assert_array_equal(sh['autocorr_time'], tau)


_NCCL_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"]); sys.path.insert(0, os.path.join(os.environ["BISIP_ROOT"], "tests"))
import numpy as np, torch, torch.distributed as dist
import bisip_b200 as bb
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=rank, world_size=world,
                        device_id=torch.device("cuda", rank))
from test_gpu_autocorr import _survey
syn = _survey("dias", 13)
kw = dict(nwalkers=32, nsteps=300, seed=11)
res = bb.fit_sharded("dias", syn["w"], syn["zn"], syn["zn_err"], discard=100, thin=2, autocorr=True, **kw)
ref = bb.BatchInversion("dias", syn["w"], syn["zn"], syn["zn_err"], **kw).fit(discard=100, thin=2, autocorr=True)
for k in ("autocorr_time", "percentiles", "mean", "std", "acceptance_fraction", "flags"):
    np.testing.assert_array_equal(res[k], ref[k])            # independent of the number of ranks
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_autocorr_two_ranks_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker_autocorr.py"
    script.write_text(_NCCL_WORKER)
    port = str(29500 + os.getpid() % 190)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out
        assert "ok" in out
