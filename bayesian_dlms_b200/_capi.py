"""ctypes binding of libbdlm.so (include/bdlm.h).  No torch types cross this boundary.

The library is loaded lazily; if it is missing, or no CUDA device is usable, every
compute entry point raises -- there is no CPU path behind this module.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BDLM_LIB_PATH") or os.path.join(HERE, "libbdlm.so")

TIME_MAJOR, SERIES_MAJOR = 0, 1
DEVICE, HOST = 0, 1
PS_V, PS_W, PS_M0, PS_C0 = 1, 2, 4, 8
PS_TIMES, PS_F, PS_G = 16, 32, 64   # Data.time / mod.f(time) / mod.g(dt) given per series
TEXTBOOK_SMOOTHER, SVD_CONSISTENT_W, PARALLEL_IN_TIME = 1, 2, 4
ST_SINGULAR, ST_NOTCONVERGED, ST_NOTPD, ST_NONFINITE, ST_TIMEOUT = 1, 2, 4, 8, 16
E_ARG, E_EMPTY, E_CUDA, E_NODEVICE, E_NCCL = -1, -2, -3, -4, -5

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)

SYMBOLS = [
    "bdlm_create", "bdlm_destroy", "bdlm_last_error", "bdlm_version", "bdlm_set_stream",
    "bdlm_sync", "bdlm_set_rng", "bdlm_launch_count", "bdlm_set_staging_bytes", "bdlm_kf_filter",
    "bdlm_rts_smooth", "bdlm_kf_filter_smooth", "bdlm_loglik", "bdlm_kf_filter_last", "bdlm_ffbs",
    "bdlm_svd_filter", "bdlm_svd_ffbs", "bdlm_gibbs_suffstats", "bdlm_wave_series",
    "bdlm_fp64_peak_tflops", "bdlm_scan_filter_smooth", "bdlm_scan_loglik", "bdlm_scan_elem_doubles",
    "bdlm_scan_combine", "bdlm_scan_ffbs",
    "bdlm_scan_dist_forward_local", "bdlm_scan_dist_forward_finish",
    "bdlm_scan_dist_backward_local", "bdlm_scan_dist_backward_finish", "bdlm_scan_dist_doubles",
    "bdlm_scan_dist_loglik_partial", "bdlm_scan_dist_loglik_finish", "bdlm_scan_dist_ffbs_local",
    "bdlm_scan_dist_ffbs_finish", "bdlm_scan_dist_ffbs_stats_finish",
    "bdlm_ar_filter", "bdlm_ar_ffbs", "bdlm_conjugate_filter", "bdlm_gibbs_draw",
    # multi-GPU communicator
    "bdlm_comm_unique_id", "bdlm_comm_create", "bdlm_comm_destroy", "bdlm_comm_last_error",
    "bdlm_comm_size", "bdlm_comm_local_size", "bdlm_comm_ctx", "bdlm_comm_sync",
    "bdlm_comm_uses_peer_exchange", "bdlm_comm_allreduce_sum", "bdlm_comm_allreduce_sum_device",
    "bdlm_comm_kf_filter", "bdlm_comm_svd_filter", "bdlm_comm_kf_filter_smooth", "bdlm_comm_loglik", "bdlm_comm_ffbs", "bdlm_comm_svd_ffbs",
    "bdlm_comm_scan_filter_smooth", "bdlm_comm_scan_loglik", "bdlm_comm_scan_ffbs",
]
# bdlm_scan_dist_doubles(n, what)
SCAN_DIST_SAMPLER_ELEM, SCAN_DIST_LOGLIK_PART, SCAN_DIST_FFBS_PART = 0, 1, 2
COMM_ID_BYTES = 128
AR1, OU = 0, 1
V_SCALAR, V_PER_STEP, V_PER_SERIES_STEP = 0, 1, 2


class Problem(C.Structure):
    _fields_ = [("B", C.c_int64), ("T", C.c_int32), ("n", C.c_int32), ("p", C.c_int32),
                ("layout", C.c_int32), ("mem", C.c_int32), ("keep_init", C.c_int32),
                ("f_tv", C.c_int32), ("g_tv", C.c_int32), ("per_series", C.c_int32),
                ("compat", C.c_int32),
                ("F", C.c_void_p), ("G", C.c_void_p), ("times", C.c_void_p),
                ("V", C.c_void_p), ("W", C.c_void_p), ("m0", C.c_void_p), ("C0", C.c_void_p),
                ("y", C.c_void_p), ("v_tv", C.c_int32), ("w_tv", C.c_int32), ("t_init", C.c_void_p)]


class KfOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("m", "C", "a", "R", "f", "Q")]


class SmoothOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("s", "S")]


class SvdOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("m", "dc", "uc", "a", "dr", "ur", "f")]


class GibbsStats(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("ssy", "ny", "ssw", "scatter")]


class ArProblem(C.Structure):
    _fields_ = [("B", C.c_int64), ("T", C.c_int32), ("layout", C.c_int32), ("mem", C.c_int32),
                ("process", C.c_int32), ("per_series", C.c_int32), ("v_mode", C.c_int32),
                ("phi", C.c_void_p), ("mu", C.c_void_p), ("sigma_eta", C.c_void_p),
                ("times", C.c_void_p), ("v", C.c_void_p), ("y", C.c_void_p)]


class ArOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("m", "C", "a", "R")]


class GibbsPrior(C.Structure):
    _fields_ = [("v_shape", C.c_double), ("v_scale", C.c_double), ("w_shape", C.c_double),
                ("w_scale", C.c_double), ("w_nu", C.c_double), ("w_psi", C.c_void_p)]


class GibbsRng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("sweep", C.c_uint64), ("gamma_v", C.c_void_p),
                ("gamma_w", C.c_void_p), ("bartlett", C.c_void_p)]


class BdlmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libbdlm error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load libbdlm.so (built in-tree by bayesian_dlms_b200.build); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m bayesian_dlms_b200.build` "
            "(the CUDA library is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.bdlm_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.bdlm_destroy.argtypes = [C.c_void_p]
    lib.bdlm_destroy.restype = None
    lib.bdlm_last_error.argtypes = [C.c_void_p]
    lib.bdlm_last_error.restype = C.c_char_p
    lib.bdlm_set_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.bdlm_sync.argtypes = [C.c_void_p]
    lib.bdlm_set_rng.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int64]
    lib.bdlm_launch_count.argtypes = [C.c_void_p]
    lib.bdlm_launch_count.restype = C.c_int64
    lib.bdlm_set_staging_bytes.argtypes = [C.c_void_p, C.c_int64]
    lib.bdlm_wave_series.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    lib.bdlm_wave_series.restype = C.c_int64
    lib.bdlm_fp64_peak_tflops.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    PP = C.POINTER(Problem)
    lib.bdlm_kf_filter.argtypes = [C.c_void_p, PP, C.POINTER(KfOut), C.c_void_p]
    lib.bdlm_rts_smooth.argtypes = [C.c_void_p, PP, C.POINTER(KfOut), C.POINTER(SmoothOut),
                                    C.c_void_p]
    lib.bdlm_kf_filter_smooth.argtypes = [C.c_void_p, PP, C.POINTER(KfOut),
                                          C.POINTER(SmoothOut), C.c_void_p]
    lib.bdlm_loglik.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bdlm_kf_filter_last.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    lib.bdlm_ffbs.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.POINTER(KfOut),
                              C.POINTER(GibbsStats), C.c_void_p]
    lib.bdlm_svd_filter.argtypes = [C.c_void_p, PP, C.POINTER(SvdOut), C.c_void_p]
    lib.bdlm_svd_ffbs.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.POINTER(SvdOut),
                                  C.POINTER(GibbsStats), C.c_void_p]
    lib.bdlm_gibbs_suffstats.argtypes = [C.c_void_p, PP, C.c_void_p, C.POINTER(GibbsStats)]
    lib.bdlm_scan_filter_smooth.argtypes = [C.c_void_p, PP, C.POINTER(KfOut),
                                            C.POINTER(SmoothOut), C.c_void_p]
    lib.bdlm_scan_loglik.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]
    lib.bdlm_scan_ffbs.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.POINTER(KfOut),
                                   C.POINTER(GibbsStats), C.c_void_p]
    lib.bdlm_scan_elem_doubles.argtypes = [C.c_int32, C.c_int32]
    lib.bdlm_scan_combine.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bdlm_scan_dist_forward_local.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_void_p]
    lib.bdlm_scan_dist_forward_finish.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_void_p,
                                                  C.POINTER(KfOut), C.c_void_p]
    lib.bdlm_scan_dist_backward_local.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32,
                                                  C.POINTER(KfOut), C.POINTER(SmoothOut), C.c_void_p]
    lib.bdlm_scan_dist_backward_finish.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_void_p,
                                                   C.POINTER(KfOut), C.POINTER(SmoothOut), C.c_void_p]
    lib.bdlm_scan_dist_doubles.argtypes = [C.c_int32, C.c_int32]
    lib.bdlm_scan_dist_loglik_partial.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
    lib.bdlm_scan_dist_loglik_finish.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]
    lib.bdlm_scan_dist_ffbs_local.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(KfOut), C.c_void_p,
                                              C.c_void_p]
    lib.bdlm_scan_dist_ffbs_finish.argtypes = [C.c_void_p, PP, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                               C.POINTER(KfOut), C.c_void_p, C.c_void_p]
    lib.bdlm_scan_dist_ffbs_stats_finish.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                                     C.POINTER(GibbsStats), C.c_void_p]
    lib.bdlm_ar_filter.argtypes = [C.c_void_p, C.POINTER(ArProblem), C.POINTER(ArOut)]
    lib.bdlm_ar_ffbs.argtypes = [C.c_void_p, C.POINTER(ArProblem), C.c_void_p, C.c_void_p,
                                 C.POINTER(ArOut)]
    lib.bdlm_conjugate_filter.argtypes = [C.c_void_p, PP, C.c_double, C.c_double,
                                          C.POINTER(KfOut), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bdlm_gibbs_draw.argtypes = [C.c_void_p, PP, C.POINTER(GibbsStats), C.POINTER(GibbsPrior),
                                    C.POINTER(GibbsRng), C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]
    lib.bdlm_comm_unique_id.argtypes = [C.c_void_p]
    lib.bdlm_comm_create.argtypes = [C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                     C.POINTER(C.c_void_p)]
    lib.bdlm_comm_destroy.argtypes = [C.c_void_p]
    lib.bdlm_comm_destroy.restype = None
    lib.bdlm_comm_last_error.argtypes = [C.c_void_p]
    lib.bdlm_comm_last_error.restype = C.c_char_p
    for name in ("bdlm_comm_size", "bdlm_comm_local_size", "bdlm_comm_sync",
                 "bdlm_comm_uses_peer_exchange"):
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.bdlm_comm_ctx.argtypes = [C.c_void_p, C.c_int32]
    lib.bdlm_comm_ctx.restype = C.c_void_p
    lib.bdlm_comm_allreduce_sum.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    lib.bdlm_comm_allreduce_sum_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    lib.bdlm_comm_kf_filter_smooth.argtypes = [C.c_void_p, PP, C.POINTER(KfOut), C.POINTER(SmoothOut),
                                               C.c_void_p]
    lib.bdlm_comm_kf_filter.argtypes = [C.c_void_p, PP, C.POINTER(KfOut), C.c_void_p]
    lib.bdlm_comm_svd_filter.argtypes = [C.c_void_p, PP, C.POINTER(SvdOut), C.c_void_p]
    lib.bdlm_comm_loglik.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bdlm_comm_ffbs.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.POINTER(KfOut),
                                   C.POINTER(GibbsStats), C.c_void_p, C.POINTER(GibbsStats)]
    lib.bdlm_comm_svd_ffbs.argtypes = [C.c_void_p, PP, C.c_void_p, C.c_void_p, C.POINTER(SvdOut),
                                       C.POINTER(GibbsStats), C.c_void_p, C.POINTER(GibbsStats)]
    lib.bdlm_comm_scan_filter_smooth.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(KfOut),
                                                 C.POINTER(SmoothOut), C.POINTER(C.c_void_p)]
    VP = C.POINTER(C.c_void_p)
    lib.bdlm_comm_scan_loglik.argtypes = [C.c_void_p, PP, VP, VP, VP, VP, VP]
    lib.bdlm_comm_scan_ffbs.argtypes = [C.c_void_p, PP, C.POINTER(C.c_int64), C.c_int64, VP, VP,
                                        C.POINTER(KfOut), C.POINTER(GibbsStats), VP]
    _lib = lib
    return lib


class Context:
    """Owns one bdlm_ctx (one GPU, one stream) -- or borrows one that a communicator owns."""

    def __init__(self, device: int = 0, borrowed_handle=None):
        lib = load()
        self._owned = borrowed_handle is None
        if self._owned:
            h = C.c_void_p()
            rc = lib.bdlm_create(int(device), C.byref(h))
            if rc != 0:
                raise BdlmError(rc, lib.bdlm_last_error(None).decode())
        else:
            h = C.c_void_p(borrowed_handle)
        self._h = h
        self.device = device
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            if self._owned:
                load().bdlm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc < 0:
            raise BdlmError(rc, load().bdlm_last_error(self._h).decode())
        return rc

    def set_stream(self, cuda_stream_handle):
        """Adopt a cudaStream_t handle (0 = legacy default stream); None = own stream."""
        if cuda_stream_handle is None:
            self.check(load().bdlm_set_stream(self._h, None, 1))
        else:
            self.check(load().bdlm_set_stream(self._h, C.c_void_p(int(cuda_stream_handle)), 0))

    def sync(self):
        self.check(load().bdlm_sync(self._h))

    def set_rng(self, seed: int, sweep: int = 0, first_series: int = 0):
        """Philox key of the FFBS calls' on-device RNG mode (z=None); ``first_series`` = global
        index of the call's first series when a batch is sharded over ranks / calls."""
        self.check(load().bdlm_set_rng(self._h, int(seed), int(sweep), int(first_series)))

    def launch_count(self) -> int:
        return int(load().bdlm_launch_count(self._h))

    def wave_series(self, n: int, p: int) -> int:
        """Series per full wave of the fused filter+smoother register kernel."""
        return int(self.check(load().bdlm_wave_series(self._h, int(n), int(p))))

    def fp64_peak_tflops(self) -> float:
        """Measured DFMA peak (TFLOP/s) of this context's GPU."""
        v = C.c_double()
        self.check(load().bdlm_fp64_peak_tflops(self._h, C.byref(v)))
        return float(v.value)

    def set_staging_bytes(self, nbytes: int):
        self.check(load().bdlm_set_staging_bytes(self._h, int(nbytes)))

    @property
    def handle(self):
        return self._h


def host_ptr(a):
    """Pointer of a C-contiguous float64 numpy array (or None)."""
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data


def make_problem(*, B, T, n, p, layout, mem, keep_init, F, G, times, V, W, m0, C0, y,
                 per_series=0, compat=0, f_tv=0, g_tv=0, v_tv=0, t_init=None, w_tv=0):
    """F, G, times: host numpy arrays (kept alive by the caller).  V, W, m0, C0, y: raw
    addresses (ints) in the memory space named by `mem`, or numpy arrays when shared."""
    pr = Problem()
    pr.B, pr.T, pr.n, pr.p = int(B), int(T), int(n), int(p)
    pr.layout, pr.mem, pr.keep_init = int(layout), int(mem), int(bool(keep_init))
    pr.f_tv, pr.g_tv, pr.per_series, pr.compat = int(f_tv), int(g_tv), int(per_series), int(compat)

    def addr(x):
        if x is None:
            return None
        return host_ptr(x) if isinstance(x, np.ndarray) else int(x)

    pr.F, pr.G, pr.times = addr(F), addr(G), addr(times)   # ints when given per series (PS_*)
    pr.V, pr.W, pr.m0, pr.C0, pr.y = addr(V), addr(W), addr(m0), addr(C0), addr(y)
    pr.v_tv = int(bool(v_tv))
    pr.w_tv = int(bool(w_tv))
    pr.t_init = addr(t_init)   # 1-element host array (kept alive by the caller) or None
    return pr
