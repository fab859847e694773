"""
ctypes binding of libvgpa_b200.so (include/vgpa_b200.h).

There is no CPU fallback: if the CUDA library has not been built the import of
this module fails loudly, and every call needs a B200 (sm_100a) device.
"""
import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["VGPA_LIB"]) if os.environ.get("VGPA_LIB") else PKG / "libvgpa_b200.so"   # override: kernel A/B runs

VGPA_OK, VGPA_EINVAL, VGPA_ENOTPD, VGPA_ECUDA = 0, 1, 2, 3
MODELS = {"DW": 0, "OU": 1, "L63": 2, "L96": 3}
METHODS = {"euler": 0, "heun": 1, "rk2": 2, "rk4": 3}
MODEL_DIM = {"DW": 1, "OU": 1, "L63": 3, "L96": 40}   # the default D; Lorenz 96 takes any 10 <= D <= 64
L96_DIMS = (10, 64)


def model_dim(key, D=None):
    """State dimension of a model: its fixed D, or for L96 the given D (default 40) checked against
    10 <= D <= 64."""
    if D is None:
        return MODEL_DIM[key]
    D = int(D)
    if key == "L96":
        if D < L96_DIMS[0]:
            raise ValueError(f" Lorenz96: Insufficient state vector dimensions: {D}")
        if D > L96_DIMS[1]:
            raise ValueError(f" Lorenz96: dim_d = {D} is outside the supported range {L96_DIMS[0]} <= dim_d <= {L96_DIMS[1]}")
    elif D != MODEL_DIM[key]:
        raise ValueError(f" {key}: state dimension {D}, expected {MODEL_DIM[key]}")
    return D

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int64)


class VgpaDesc(C.Structure):
    _fields_ = [("model", C.c_int32), ("method", C.c_int32), ("D", C.c_int32), ("N", C.c_int32),
                ("M", C.c_int32), ("B", C.c_int32), ("device", C.c_int32), ("reserved", C.c_int32),
                ("dt", C.c_double), ("dt_model", C.c_double),
                ("theta", _dp), ("theta_stride", C.c_int64),
                ("sigma", _dp), ("sigma_stride", C.c_int64),
                ("R", _dp), ("R_stride", C.c_int64),
                ("obs_t", _ip),
                ("obs_y", _dp), ("obs_y_stride", C.c_int64),
                ("m0", _dp), ("m0_stride", C.c_int64),
                ("s0", _dp), ("s0_stride", C.c_int64),
                ("E0", _dp), ("E0_stride", C.c_int64),
                ("scratch_bytes", C.c_int64)]


class VgpaFullOut(C.Structure):
    _fields_ = [(k, _dp) for k in ("F", "parts", "grad", "mt", "st", "lamt", "psit", "Efx", "Edf",
                                   "dEsde_dm", "dEsde_ds")]


def _load():
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library has not been built. Run "
            "`python -m vgpa_b200.build` (needs nvcc; cross-compiles without a GPU). "
            "vgpa_b200 has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    H = C.c_void_p
    lib.vgpa_create.restype = C.c_int
    lib.vgpa_create.argtypes = [C.POINTER(VgpaDesc), C.POINTER(H)]
    lib.vgpa_create_obs_rows.restype = C.c_int
    lib.vgpa_create_obs_rows.argtypes = [C.POINTER(VgpaDesc), C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(H)]
    lib.vgpa_create_observed.restype = C.c_int
    lib.vgpa_create_observed.argtypes = [C.POINTER(VgpaDesc), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.POINTER(H)]
    lib.vgpa_destroy.restype = None
    lib.vgpa_destroy.argtypes = [H]
    lib.vgpa_last_error.restype = C.c_char_p
    lib.vgpa_last_error.argtypes = [H]
    lib.vgpa_eval.restype = C.c_int
    lib.vgpa_eval.argtypes = [H, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
    lib.vgpa_eval_device.restype = C.c_int
    lib.vgpa_eval_device.argtypes = [H, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_int64, C.c_void_p]
    lib.vgpa_hyper_device.restype = C.c_int
    lib.vgpa_hyper_device.argtypes = [H, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                      C.c_void_p, C.c_int64, C.c_void_p]
    lib.vgpa_initialization.restype = C.c_int
    lib.vgpa_initialization.argtypes = [H, C.c_double, C.c_void_p, C.c_int64, C.c_void_p]
    lib.vgpa_initialization_host.restype = C.c_int
    lib.vgpa_initialization_host.argtypes = [H, C.c_double, _dp, C.c_int64]
    lib.vgpa_sync.restype = C.c_int
    lib.vgpa_sync.argtypes = [H]
    lib.vgpa_set_active.restype = C.c_int
    lib.vgpa_set_active.argtypes = [H, C.c_void_p]
    lib.vgpa_set_active_list.restype = C.c_int
    lib.vgpa_set_active_list.argtypes = [H, C.c_void_p, C.c_int32]
    lib.vgpa_eval_full.restype = C.c_int
    lib.vgpa_eval_full.argtypes = [H, C.c_int64, _dp, C.POINTER(VgpaFullOut)]
    lib.vgpa_solve_fwd.restype = C.c_int
    lib.vgpa_solve_fwd.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double] + [_dp] * 7
    lib.vgpa_solve_bwd.restype = C.c_int
    lib.vgpa_solve_bwd.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double] + [_dp] * 7
    lib.vgpa_model_energy.restype = C.c_int
    lib.vgpa_model_energy.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double] + [_dp] * 13
    lib.vgpa_obs_energy.restype = C.c_int
    lib.vgpa_obs_energy.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _ip] + [_dp] * 8
    lib.vgpa_obs_energy_observed.restype = C.c_int
    lib.vgpa_obs_energy_observed.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, C.c_uint64] + [_dp] * 5
    i64 = C.c_int64
    traj = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double] + [C.c_void_p, i64] * 5
    obs = [C.c_int] * 5 + [C.c_void_p] + [C.c_void_p, i64] * 4
    traj_dim = traj[:2] + [C.c_int] + traj[2:]
    for name, args in (("vgpa_make_trajectory", traj), ("vgpa_make_trajectory_device", traj + [C.c_void_p]),
                       ("vgpa_make_trajectory_dim", traj_dim),
                       ("vgpa_make_trajectory_device_dim", traj_dim + [C.c_void_p]),
                       ("vgpa_collect_obs", obs), ("vgpa_collect_obs_device", obs + [C.c_void_p])):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    lib.vgpa_host_alloc.restype = C.c_void_p
    lib.vgpa_host_alloc.argtypes = [C.c_int64]
    lib.vgpa_scratch_cache.restype = C.c_longlong
    lib.vgpa_scratch_cache.argtypes = [C.c_int]
    lib.vgpa_host_free.restype = None
    lib.vgpa_host_free.argtypes = [C.c_void_p]
    lib.vgpa_host_copy.restype = None
    lib.vgpa_host_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
    lib.vgpa_host_equal.restype = C.c_int
    lib.vgpa_host_equal.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
    lib.vgpa_launch_count.restype = C.c_int64
    lib.vgpa_launch_count.argtypes = [H]
    lib.vgpa_chunk_size.restype = C.c_int64
    lib.vgpa_chunk_size.argtypes = [H]
    lib.vgpa_scratch_in_use.restype = C.c_int64
    lib.vgpa_scratch_in_use.argtypes = [H]
    lib.vgpa_set_timing.restype = C.c_int
    lib.vgpa_set_timing.argtypes = [H, C.c_int]
    lib.vgpa_get_timing.restype = C.c_int
    lib.vgpa_get_timing.argtypes = [H, _dp, _ip]
    vp, i32p = C.c_void_p, C.c_void_p
    for name, args in (("vgpa_bdot", [C.c_int, C.c_int64, vp, vp, vp, C.c_int64, vp, i32p, vp]),
                       ("vgpa_baxpy", [C.c_int, C.c_int64, vp, vp, vp, vp, C.c_int64, i32p, vp]),
                       ("vgpa_bdir", [C.c_int, C.c_int64, i32p, vp, vp, vp, C.c_int64, vp]),
                       ("vgpa_bcopy", [C.c_int, C.c_int64, i32p, vp, vp, C.c_int64, vp]),
                       ("vgpa_bstats", [C.c_int, C.c_int64, vp, C.c_int64, vp, i32p, vp])):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    lib.vgpa_version.restype = C.c_char_p
    return lib


lib = _load()


def raise_for(rc, handle=None):
    """Map a library return code to the exception the reference would raise."""
    if rc == VGPA_OK:
        return
    msg = lib.vgpa_last_error(handle).decode("utf-8", "replace")
    if rc == VGPA_EINVAL:
        raise ValueError(msg)
    if rc == VGPA_ENOTPD:
        raise np.linalg.LinAlgError(msg)   # numpy.linalg.cholesky in utilities.py:211,275
    raise RuntimeError(msg)


def dptr(a):
    return a.ctypes.data_as(_dp)


def f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


class PinnedArray:
    """A numpy float64 array over page-locked host memory (vgpa_host_alloc)."""

    def __init__(self, shape):
        n = int(np.prod(shape))
        self._ptr = lib.vgpa_host_alloc(max(n, 1) * 8)
        if not self._ptr:
            raise MemoryError(f"vgpa_host_alloc({n * 8}) failed")
        buf = (C.c_double * max(n, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=np.float64, count=n).reshape(shape)

    def free(self):
        if self._ptr:
            self.array = None
            lib.vgpa_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
