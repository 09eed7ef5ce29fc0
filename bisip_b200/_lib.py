"""ctypes binding of ``csrc/libbisip_b200.so`` (the C ABI in ``include/bisip_b200.h``).

PyTorch is used only for device memory, streams and ``torch.distributed``; every hot-path
computation goes through the ``extern "C"`` entry points bound here.  There is NO CPU
fallback: a missing library or a missing CUDA device raises immediately.
"""
import ctypes as C
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BISIP_B200_LIB", os.path.join(_HERE, "csrc", "libbisip_b200.so"))   # env: developer builds

MODEL_COLECOLE, MODEL_DIAS, MODEL_SHIN, MODEL_DECOMP = 0, 1, 2, 3
PREC_FP64, PREC_TF32, PREC_3XTF32, PREC_TF32_MMA, PREC_3XTF32_MMA, PREC_FP64_COLLAPSED = 0, 1, 2, 3, 4, 5
PRECISIONS = {"fp64": PREC_FP64, "tf32": PREC_TF32, "3xtf32": PREC_3XTF32,
              "tf32-mma": PREC_TF32_MMA, "3xtf32-mma": PREC_3XTF32_MMA, "fp64-collapsed": PREC_FP64_COLLAPSED}
MAX_PCT = 16
ABI_VERSION = 2

EXPORTS = ("bisip_abi_version", "bisip_last_error", "bisip_launch_count", "bisip_forward",
           "bisip_log_probability", "bisip_decomp_build_kernel", "bisip_n_keep",
           "bisip_ensemble_run", "bisip_column_stats_workspace", "bisip_column_stats",
           "bisip_decomp_kernel_kind", "bisip_model_percentile", "bisip_gauss_loglike",
           "bisip_autocorr_time", "bisip_rtd_stats")
KERNEL_KINDS = {0: "dmma", 1: "dmma-cluster", 2: "mma-tf32", 3: "tcgen05", 4: "tcgen05-cluster", 5: "fp64-collapsed"}


class BisipError(RuntimeError):
    pass


class ModelDesc(C.Structure):
    _fields_ = [("model", C.c_int32), ("ndim", C.c_int32), ("n_freq", C.c_int32),
                ("n_modes", C.c_int32), ("n_tau", C.c_int32), ("n_coef", C.c_int32),
                ("precision", C.c_int32), ("reserved", C.c_int32), ("c_exp", C.c_double)]


_lib = None


def load():
    """Load the shared library (no GPU needed to load it or to resolve its symbols)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BisipError(
            f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "bisip_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.bisip_abi_version.restype = C.c_int
    lib.bisip_last_error.restype = C.c_char_p
    lib.bisip_launch_count.restype = C.c_int64
    lib.bisip_n_keep.restype = C.c_int
    lib.bisip_n_keep.argtypes = [C.c_int, C.c_int, C.c_int]
    vp, i32, i64, dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
    lib.bisip_forward.restype = C.c_int
    lib.bisip_forward.argtypes = [C.POINTER(ModelDesc), i32, i32, vp, vp, i64, vp, vp, i64, vp, vp]
    lib.bisip_log_probability.restype = C.c_int
    lib.bisip_log_probability.argtypes = [C.POINTER(ModelDesc), i32, i32, vp, vp, i64, vp, vp, i64,
                                          vp, vp, vp, vp, vp]
    lib.bisip_decomp_build_kernel.restype = C.c_int
    lib.bisip_decomp_build_kernel.argtypes = [vp, i32, vp, i32, dbl, vp, vp]
    lib.bisip_gauss_loglike.restype = C.c_int
    lib.bisip_gauss_loglike.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.bisip_ensemble_run.restype = C.c_int
    lib.bisip_ensemble_run.argtypes = [C.POINTER(ModelDesc), i32, i32, i32, i32, C.c_uint64, C.c_uint32,
                                       dbl, i32, i32, vp, i64, vp, vp, i64, vp, vp, vp,
                                       vp, vp, vp, vp, vp, vp, vp]
    lib.bisip_decomp_kernel_kind.restype = C.c_int
    lib.bisip_decomp_kernel_kind.argtypes = [C.POINTER(ModelDesc), i32]
    lib.bisip_column_stats_workspace.restype = C.c_int64
    lib.bisip_column_stats_workspace.argtypes = [i32, i64, i32]
    lib.bisip_column_stats.restype = C.c_int
    lib.bisip_column_stats.argtypes = [vp, i32, i64, i32, i32, C.POINTER(C.c_int64), C.POINTER(C.c_double),
                                       vp, vp, vp, vp, i64, vp]
    lib.bisip_model_percentile.restype = C.c_int
    lib.bisip_model_percentile.argtypes = [C.POINTER(ModelDesc), i32, i64, vp, vp, i64, vp, vp, i64, i32,
                                           C.POINTER(C.c_int64), C.POINTER(C.c_double), vp, vp]
    lib.bisip_autocorr_time.restype = C.c_int
    lib.bisip_autocorr_time.argtypes = [vp, i32, i32, i32, i32, dbl, vp, vp]
    lib.bisip_rtd_stats.restype = C.c_int
    lib.bisip_rtd_stats.argtypes = [i32, i64, i32, i32, i32, vp, vp, i64, i32, C.POINTER(C.c_int64),
                                    C.POINTER(C.c_double), vp, vp, vp, vp]
    if lib.bisip_abi_version() != ABI_VERSION:
        raise BisipError("libbisip_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().bisip_last_error()
        raise BisipError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")


def launch_count():
    return int(load().bisip_launch_count())


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise BisipError("bisip_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")


def dev_f64(a, device):
    """Host array / tensor -> contiguous float64 device tensor."""
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64))).to(device)


_CONST_CACHE = {}
_CONST_CACHE_MAX = 128


def dev_const(a, device):
    """Device copy of a small read-only host array (w, zn, zn_err, taus, log_taus, bounds), cached by content:
    the single-spectrum API (``forward`` / ``_log_probability`` called in a loop, e.g. by an optimiser) would
    otherwise re-upload the same constants on every call.  The cached tensors must not be written to."""
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64).contiguous()
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if a.nbytes > (1 << 16):
        return torch.from_numpy(a).to(device)
    key = (str(device), a.shape, a.tobytes())
    t = _CONST_CACHE.get(key)
    if t is None:
        if len(_CONST_CACHE) >= _CONST_CACHE_MAX:
            _CONST_CACHE.pop(next(iter(_CONST_CACHE)))
        t = torch.from_numpy(a).to(device)
        _CONST_CACHE[key] = t
    return t


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def percentile_indices(n, p):
    """Virtual index of NumPy's default 'linear' percentile, computed with NumPy's own
    arithmetic (numpy/lib/_function_base_impl.py: q = p/100; (n-1)*q; floor; gamma)."""
    q = np.true_divide(np.asanyarray(p, dtype=np.float64), 100)
    if not (np.all(q >= 0) and np.all(q <= 1)):
        raise ValueError("Percentiles must be in the range [0, 100]")
    virt = np.asanyarray((n - 1) * q)
    lo = np.floor(virt)
    gamma = virt - lo
    return np.atleast_1d(lo).astype(np.int64), np.atleast_1d(gamma).astype(np.float64)
