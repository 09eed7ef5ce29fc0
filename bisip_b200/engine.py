"""Device-side entry points: thin tensor wrappers over the C ABI (``include/bisip_b200.h``).

Everything here takes / returns CUDA float64 tensors and launches on torch's current
stream.  Shapes follow the reference's conventions: parameter vectors ``theta`` are ordered
like the reference's ``params`` dicts (reference ``models.py:212-213, 249-252, 287-291,
325-331``); spectra are ``(2, N)`` arrays with rows ``[real; imag]`` (``utils.py:141-142``).
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib


@dataclass
class ModelSpec:
    """Model constants shared by a batch of spectra."""
    model: int                      # _lib.MODEL_*
    ndim: int
    n_modes: int = 1                # ColeCole
    taus: torch.Tensor = None       # Decomp: (S,) or (B,S)
    log_taus: torch.Tensor = None   # Decomp: (D,S) or (B,D,S)
    c_exp: float = 1.0
    precision: int = _lib.PREC_FP64

    def desc(self, n_freq):
        n_tau = int(self.taus.shape[-1]) if self.taus is not None else 0
        n_coef = int(self.log_taus.shape[-2]) if self.log_taus is not None else 0
        return _lib.ModelDesc(self.model, self.ndim, int(n_freq), int(self.n_modes), n_tau, n_coef,
                              int(self.precision), 0, float(self.c_exp))

    def tau_stride(self):
        if self.taus is None or self.taus.dim() == 1:
            return 0
        return int(self.taus.shape[-1])


def _w_stride(w):
    return 0 if w.dim() == 1 else int(w.shape[-1])


def _chk_cuda_f64(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
            raise _lib.BisipError("engine tensors must be contiguous CUDA float64")


def decomp_kernel_kind(spec, n_freq, n_walkers):
    """Name of the decomposition kernel ``ensemble_run`` will launch for this model spec and walker count:
    'dmma', 'dmma-cluster', 'mma-tf32' or 'tcgen05' (needs a CUDA device: the answer depends on its shared memory)."""
    lib = _lib.load()
    d = spec.desc(n_freq)
    rc = lib.bisip_decomp_kernel_kind(C.byref(d), int(n_walkers))
    if rc < 0:
        _lib.check(rc, "bisip_decomp_kernel_kind")
    return _lib.KERNEL_KINDS[rc]


def forward(spec, theta, w):
    """theta (B, n, ndim), w (N,) or (B, N)  ->  Z (B, n, 2, N).  Reference: Model.forward."""
    lib = _lib.load()
    _chk_cuda_f64(theta, w, spec.taus, spec.log_taus)
    B, n, ndim = theta.shape
    N = w.shape[-1]
    assert ndim == spec.ndim
    Z = torch.empty((B, n, 2, N), dtype=torch.float64, device=theta.device)
    d = spec.desc(N)
    rc = lib.bisip_forward(C.byref(d), B, n, _lib.ptr(theta), _lib.ptr(w), _w_stride(w),
                           _lib.ptr(spec.taus), _lib.ptr(spec.log_taus), spec.tau_stride(),
                           _lib.ptr(Z), _lib.stream_ptr(theta.device))
    _lib.check(rc, "bisip_forward")
    return Z


def log_probability(spec, theta, w, y, yerr, bounds):
    """theta (B, n, ndim); y, yerr (B, 2, N); bounds (2, ndim) -> lp (B, n).
    Reference: Inversion._log_probability (models.py:71-76)."""
    lib = _lib.load()
    _chk_cuda_f64(theta, w, y, yerr, bounds, spec.taus, spec.log_taus)
    B, n, ndim = theta.shape
    N = w.shape[-1]
    lp = torch.empty((B, n), dtype=torch.float64, device=theta.device)
    d = spec.desc(N)
    rc = lib.bisip_log_probability(C.byref(d), B, n, _lib.ptr(theta), _lib.ptr(w), _w_stride(w),
                                   _lib.ptr(spec.taus), _lib.ptr(spec.log_taus), spec.tau_stride(),
                                   _lib.ptr(y), _lib.ptr(yerr), _lib.ptr(bounds), _lib.ptr(lp),
                                   _lib.stream_ptr(theta.device))
    _lib.check(rc, "bisip_log_probability")
    return lp


def gauss_loglike(Z, y, yerr):
    """Z (n, 2, N) caller-supplied model rows; y, yerr (2, N) -> ll (n,).
    Reference: Inversion._log_likelihood with a user callable (models.py:59-62)."""
    lib = _lib.load()
    _chk_cuda_f64(Z, y, yerr)
    n, N = Z.shape[0], Z.shape[-1]
    ll = torch.empty((n,), dtype=torch.float64, device=Z.device)
    rc = lib.bisip_gauss_loglike(_lib.ptr(Z), _lib.ptr(y), _lib.ptr(yerr), N, n, _lib.ptr(ll),
                                 _lib.stream_ptr(Z.device))
    _lib.check(rc, "bisip_gauss_loglike")
    return ll


def decomp_kernel_matrix(w, taus, c_exp):
    """K (S, 2N) = 1 - 1/(1+(i w tau)^c): columns [real | imag]."""
    lib = _lib.load()
    _chk_cuda_f64(w, taus)
    N, S = w.shape[0], taus.shape[0]
    K = torch.empty((S, 2 * N), dtype=torch.float64, device=w.device)
    rc = lib.bisip_decomp_build_kernel(_lib.ptr(w), N, _lib.ptr(taus), S, float(c_exp), _lib.ptr(K),
                                       _lib.stream_ptr(w.device))
    _lib.check(rc, "bisip_decomp_build_kernel")
    return K


def n_keep(nsteps, discard=0, thin=1):
    return int(_lib.load().bisip_n_keep(int(nsteps), int(discard), int(thin)))


def ensemble_run(spec, coords, w, y, yerr, bounds, nsteps, seed, spectrum0=0, a=2.0, discard=0,
                 thin=1, step0=0, store_chain=True, store_logp=True):
    """Run the on-device stretch-move sampler for a batch of spectra.

    coords (B, W, ndim) is updated in place (p0 -> final ensemble).  Returns a dict with
    chain (B, n_keep, W, ndim) | None, log_prob (B, n_keep, W) | None, lp (B, W),
    accepted (B, W) int32, flags (B,) int32.
    """
    lib = _lib.load()
    _chk_cuda_f64(coords, w, y, yerr, bounds, spec.taus, spec.log_taus)
    B, W, ndim = coords.shape
    N = w.shape[-1]
    dev = coords.device
    nk = n_keep(nsteps, discard, thin)
    chain = torch.empty((B, nk, W, ndim), dtype=torch.float64, device=dev) if store_chain else None
    logp = torch.empty((B, nk, W), dtype=torch.float64, device=dev) if store_logp else None
    lp = torch.empty((B, W), dtype=torch.float64, device=dev)
    accepted = torch.empty((B, W), dtype=torch.int32, device=dev)
    flags = torch.empty((B,), dtype=torch.int32, device=dev)
    d = spec.desc(N)
    rc = lib.bisip_ensemble_run(C.byref(d), B, W, int(nsteps), int(step0), C.c_uint64(int(seed) & (2**64 - 1)),
                                C.c_uint32(int(spectrum0) & 0xffffffff), float(a), int(discard), int(thin),
                                _lib.ptr(w), _w_stride(w), _lib.ptr(spec.taus), _lib.ptr(spec.log_taus),
                                spec.tau_stride(), _lib.ptr(y), _lib.ptr(yerr), _lib.ptr(bounds),
                                _lib.ptr(coords), _lib.ptr(lp), _lib.ptr(chain), _lib.ptr(logp),
                                _lib.ptr(accepted), _lib.ptr(flags), _lib.stream_ptr(dev))
    _lib.check(rc, "bisip_ensemble_run")
    return dict(chain=chain, log_prob=logp, lp=lp, accepted=accepted, flags=flags, coords=coords)


def column_stats(data, p=None, want_mean=False, want_std=False):
    """data (B, n, ncol) -> dict(pct (B, len(p), ncol), mean (B, ncol), std (B, ncol)).
    Exact NumPy-'linear' percentiles, mean and population std over axis 1; ``data`` is read in place."""
    lib = _lib.load()
    _chk_cuda_f64(data)
    B, n, ncol = data.shape
    dev = data.device
    out = {}
    p_arr = np.atleast_1d(np.asarray(p, dtype=np.float64)) if p is not None else np.empty(0)
    npct = int(p_arr.shape[0])
    mean = torch.empty((B, ncol), dtype=torch.float64, device=dev) if want_mean else None
    std = torch.empty((B, ncol), dtype=torch.float64, device=dev) if want_std else None
    pct = torch.empty((B, npct, ncol), dtype=torch.float64, device=dev) if npct else None
    done_stats = False
    for s0 in range(0, max(npct, 1), _lib.MAX_PCT):
        pp = p_arr[s0:s0 + _lib.MAX_PCT]
        k = int(pp.shape[0])
        whole = k == npct                      # the usual case: the kernel writes straight into the result
        if k:
            lo, gamma = _lib.percentile_indices(n, pp)
            lo_c = (C.c_int64 * k)(*[int(v) for v in lo])
            ga_c = (C.c_double * k)(*[float(v) for v in gamma])
            part = pct if whole else torch.empty((B, k, ncol), dtype=torch.float64, device=dev)
        else:
            lo_c = ga_c = None
            part = None
        rc = lib.bisip_column_stats(_lib.ptr(data), B, n, ncol, k, lo_c, ga_c, _lib.ptr(part),
                                    _lib.ptr(mean if not done_stats else None),
                                    _lib.ptr(std if not done_stats else None),
                                    None, 0, _lib.stream_ptr(dev))
        _lib.check(rc, "bisip_column_stats")
        done_stats = True
        if k and not whole:
            pct[:, s0:s0 + k] = part
    out["pct"], out["mean"], out["std"] = pct, mean, std
    return out


def autocorr_time(chain, c=5.0):
    """emcee's integrated autocorrelation time of every column: chain (B, n_keep, W, ncol) -> (B, ncol), in steps of
    the kept chain (``bisip_autocorr_time``; the chain is read in place).  A column with a constant walker or a NaN
    gives NaN."""
    lib = _lib.load()
    _chk_cuda_f64(chain)
    B, nk, W, ncol = chain.shape
    dev = chain.device
    out = torch.empty((B, ncol), dtype=torch.float64, device=dev)
    for s0 in range(0, B, 65535):                  # one launch per 65,535 spectra (grid y)
        k = min(65535, B - s0)
        rc = lib.bisip_autocorr_time(_lib.ptr(chain[s0:s0 + k]), k, nk, W, ncol, float(c), _lib.ptr(out[s0:s0 + k]),
                                     _lib.stream_ptr(dev))
        _lib.check(rc, "bisip_autocorr_time")
    return out


def rtd_stats(theta, log_taus, p=None, want_mean=False, want_std=False):
    """Relaxation-time distribution and total chargeability of a decomposition over parameter vectors
    (``bisip_rtd_stats``; ``theta`` is read in place): theta (B, n, 1 + n_coef), log_taus (n_coef, n_tau) or
    (B, n_coef, n_tau) -> dict(pct (B, len(p), n_tau + 1), mean (B, n_tau + 1), std (B, n_tau + 1)).  Columns
    [0, n_tau) are the RTD m_l = sum_i a_i log_taus[i, l], equal to ``products.relaxation_time_distribution`` bit for
    bit; column n_tau is the total chargeability sum_l m_l.  Statistics over axis 1 as ``column_stats``."""
    lib = _lib.load()
    _chk_cuda_f64(theta, log_taus)
    B, n, ndim = theta.shape
    n_coef, n_tau = int(log_taus.shape[-2]), int(log_taus.shape[-1])
    if ndim != 1 + n_coef:
        raise ValueError(f"expected {n_coef} coefficients, got {ndim - 1}")
    tau_stride = 0 if log_taus.dim() == 2 else n_tau
    dev = theta.device
    p_arr = np.atleast_1d(np.asarray(p, dtype=np.float64)) if p is not None else np.empty(0)
    npct = int(p_arr.shape[0])
    C_out = n_tau + 1
    pct = torch.empty((B, npct, C_out), dtype=torch.float64, device=dev) if npct else None
    mean = torch.empty((B, C_out), dtype=torch.float64, device=dev) if want_mean else None
    std = torch.empty((B, C_out), dtype=torch.float64, device=dev) if want_std else None
    chunks = [(q0, p_arr[q0:q0 + _lib.MAX_PCT]) for q0 in range(0, npct, _lib.MAX_PCT)] or [(0, p_arr)]
    for s0 in range(0, B, 65535):                  # one launch per 65,535 spectra (grid y) and 16 percentiles
        k = min(65535, B - s0)
        lt = log_taus if tau_stride == 0 else log_taus[s0:s0 + k]
        for i, (q0, pp) in enumerate(chunks):
            m = int(pp.shape[0])
            if m:
                lo, gamma = _lib.percentile_indices(n, pp)
                lo_c = (C.c_int64 * m)(*[int(v) for v in lo])
                ga_c = (C.c_double * m)(*[float(v) for v in gamma])
                whole = m == npct and k == B           # the usual case: the kernel writes straight into the result
                part = pct if whole else torch.empty((k, m, C_out), dtype=torch.float64, device=dev)
            else:
                lo_c = ga_c = part = None
            first = i == 0                         # mean / std with the first percentile block only
            rc = lib.bisip_rtd_stats(k, n, ndim, n_coef, n_tau, _lib.ptr(theta[s0:s0 + k]), _lib.ptr(lt), tau_stride,
                                     m, lo_c, ga_c, _lib.ptr(part),
                                     _lib.ptr(mean[s0:s0 + k] if first and want_mean else None),
                                     _lib.ptr(std[s0:s0 + k] if first and want_std else None), _lib.stream_ptr(dev))
            _lib.check(rc, "bisip_rtd_stats")
            if m and not whole:
                pct[s0:s0 + k, q0:q0 + m] = part
    return {"pct": pct, "mean": mean, "std": std}


def model_percentile(spec, theta, w, p):
    """Percentiles of the forward model over parameter vectors, fused (``bisip_model_percentile``): theta (B, n, ndim),
    w (N,) or (B, N), p percentiles -> (B, len(p), 2, N).  The (n, 2N) model matrix is never materialised.  Returns None
    when n exceeds what one CTA's shared memory holds (the caller composes ``forward`` + ``column_stats``)."""
    lib = _lib.load()
    _chk_cuda_f64(theta, w, spec.taus, spec.log_taus)
    B, n, ndim = theta.shape
    N = w.shape[-1]
    dev = theta.device
    p_arr = np.atleast_1d(np.asarray(p, dtype=np.float64))
    npct = int(p_arr.shape[0])
    out = torch.empty((B, npct, 2, N), dtype=torch.float64, device=dev)
    d = spec.desc(N)
    for s0 in range(0, npct, _lib.MAX_PCT):
        pp = p_arr[s0:s0 + _lib.MAX_PCT]
        k = int(pp.shape[0])
        lo, gamma = _lib.percentile_indices(n, pp)
        lo_c = (C.c_int64 * k)(*[int(v) for v in lo])
        ga_c = (C.c_double * k)(*[float(v) for v in gamma])
        part = out if k == npct else torch.empty((B, k, 2, N), dtype=torch.float64, device=dev)
        rc = lib.bisip_model_percentile(C.byref(d), B, n, _lib.ptr(theta), _lib.ptr(w), _w_stride(w),
                                        _lib.ptr(spec.taus), _lib.ptr(spec.log_taus), spec.tau_stride(), k, lo_c, ga_c,
                                        _lib.ptr(part), _lib.stream_ptr(dev))
        if rc == -2 and "shared memory" in (lib.bisip_last_error() or b"").decode():
            return None
        _lib.check(rc, "bisip_model_percentile")
        if k != npct:
            out[:, s0:s0 + k] = part
    return out
