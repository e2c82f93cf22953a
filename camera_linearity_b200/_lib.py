"""ctypes binding of the C ABI declared in ``include/camera_linearity.h``.

There is no CPU fallback: if ``libcamlin_b200.so`` is missing (and cannot be built because nvcc
is absent) importing the ops raises.  The library is kept in-tree next to this file.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libcamlin_b200.so"

CL_MAX_EXPOSURES = 32
CL_MAX_CHANNELS = 8
CL_MAX_MEDIAN_KERNEL = 7
CL_MAX_PAIR_EXPOSURES = 8

_STATUS_NAMES = {0: "CL_OK", -1: "CL_ERR_INVALID_ARGUMENT", -2: "CL_ERR_UNSUPPORTED",
                 -3: "CL_ERR_WORKSPACE", -4: "CL_ERR_ALIGNMENT"}


class CamlinError(RuntimeError):
    def __init__(self, status: int, what: str, message: str):
        super().__init__(f"{what} failed: {_STATUS_NAMES.get(status, status)} ({message})")
        self.status = status


class HdrMergeArgs(C.Structure):
    """``cl_hdr_merge_args`` (include/camera_linearity.h)."""
    _fields_ = [
        ("n_exposures", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
        ("channels", C.c_int32), ("dn_bytes", C.c_int32), ("bits", C.c_int32),
        ("dn", C.POINTER(C.c_void_p)), ("std", C.POINTER(C.c_void_p)),
        ("exposure_s", C.POINTER(C.c_double)),
        ("lut", C.c_void_p), ("dlut", C.c_void_p), ("std_lut", C.c_void_p),
        ("dark", C.POINTER(C.c_void_p)), ("dark_scale", C.POINTER(C.c_double)),
        ("dark_threshold", C.c_double), ("median_kernel", C.c_int32), ("flat_bytes", C.c_int32),
        ("flat", C.c_void_p), ("flat_std", C.c_void_p), ("flat_means", C.c_void_p),
        ("out_val", C.c_void_p), ("out_std", C.c_void_p),
        ("algo", C.c_int32), ("reserved", C.c_int32),
    ]


class IcrfProblem(C.Structure):
    """``cl_icrf_problem`` (include/camera_linearity.h)."""
    _fields_ = [
        ("n_candidates", C.c_int32), ("n_params", C.c_int32), ("datapoints", C.c_int32),
        ("use_mean_icrf", C.c_int32), ("lower", C.c_int32), ("upper", C.c_int32),
        ("n_exposures", C.c_int32), ("use_std", C.c_int32),
    ]


CL_MAX_PEERS = 16


class PeerGroup(C.Structure):
    """``cl_peer_group`` (include/camera_linearity.h)."""
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("buffers", C.c_void_p * CL_MAX_PEERS)]


class DeSelectArgs(C.Structure):
    """``cl_de_select_args`` (include/camera_linearity.h)."""
    _fields_ = [("pop", C.c_void_p), ("energies", C.c_void_p), ("trial", C.c_void_p), ("n_members", C.c_int32),
                ("n_params", C.c_int32), ("tol", C.c_double), ("atol", C.c_double), ("generation", C.c_void_p),
                ("status", C.c_void_p), ("best", C.c_void_p)]


class IpcHandle(C.Structure):
    """``cl_ipc_handle`` (include/camera_linearity.h)."""
    _fields_ = [("bytes", C.c_ubyte * 64)]


_vp, _i, _i64, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_size_t

# name -> (restype, argtypes); every symbol include/camera_linearity.h declares
SIGNATURES = {
    "cl_abi_version": (_i, []),
    "cl_status_string": (C.c_char_p, [_i]),
    "cl_launch_count": (C.c_uint64, []),
    "cl_linearize_dn": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "cl_linearize_f64": (_i, [_vp, _d, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "cl_hdr_merge_workspace_bytes": (_sz, [C.POINTER(HdrMergeArgs)]),
    "cl_hdr_merge": (_i, [C.POINTER(HdrMergeArgs), _vp, _sz, _vp]),
    "cl_flat_roi_means_workspace_bytes": (_sz, [_i, _i, _i]),
    "cl_flat_roi_means": (_i, [_vp, _i, _d, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "cl_gaussian_weight": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "cl_bad_pixel_filter": (_i, [_vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp, _vp]),
    "cl_flat_field_normalize": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _vp, _vp, _vp]),
    "cl_welford_update": (_i, [_vp, _i, _i64, _i, _vp, _d, _vp, _vp, _i64, _vp]),
    "cl_welford_finalize": (_i, [_vp, _vp, _i64, _i64, _d, _vp, _vp, _vp]),
    "cl_welford_stack_workspace_bytes": (_sz, [_i, _i64]),
    "cl_welford_stack": (_i, [_vp, _i, _i64, _i, _vp, _d, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cl_welford_update_u16": (_i, [_vp, _i, _i64, _i, _vp, _i, _d, _vp, _vp, _i64, _vp]),
    "cl_welford_finalize_u16": (_i, [_vp, _vp, _i64, _i64, _d, _vp, _vp, _vp]),
    "cl_welford_stack_u16": (_i, [_vp, _i, _i64, _i, _vp, _i, _d, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cl_icrf_tables_bytes": (_sz, [C.POINTER(IcrfProblem)]),
    "cl_icrf_curves": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cl_icrf_energy_workspace_bytes": (_sz, [C.POINTER(IcrfProblem), _i64]),
    "cl_icrf_energy_partial": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, C.POINTER(C.c_double),
                                    _i64, _vp, _vp, _sz, _vp]),
    "cl_icrf_energy_partial_u16": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, C.POINTER(C.c_double),
                                        _i64, _vp, _vp, _sz, _vp]),
    "cl_icrf_energy_finalize": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, _vp]),
    "cl_icrf_exchange_bytes": (_sz, [C.POINTER(IcrfProblem), _i]),
    "cl_icrf_energy_population": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, C.POINTER(C.c_double), _i64, _vp, _vp,
                                       _vp, _vp, _sz, C.POINTER(PeerGroup), C.POINTER(DeSelectArgs), _vp]),
    "cl_icrf_energy_population_u16": (_i, [C.POINTER(IcrfProblem), _vp, _vp, _vp, C.POINTER(C.c_double), _i64, _vp,
                                           _vp, _vp, _vp, _sz, C.POINTER(PeerGroup), C.POINTER(DeSelectArgs), _vp]),
    "cl_peer_alloc": (_i, [_sz, C.POINTER(C.c_void_p), C.POINTER(IpcHandle)]),
    "cl_peer_open": (_i, [C.POINTER(IpcHandle), C.POINTER(C.c_void_p)]),
    "cl_peer_close": (_i, [_vp]),
    "cl_peer_free": (_i, [_vp]),
    "cl_de_trial_curves": (_i, [C.POINTER(IcrfProblem), _vp, _i, _d, _d, _d, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp, _vp, _vp]),
    "cl_measurand_binary": (_i, [_i, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "cl_measurand_log": (_i, [_i, _vp, _vp, _i64, _vp, _vp, _vp]),
    "cl_measurand_difference": (_i, [_vp, _vp, _vp, _vp, _d, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cl_noise_profiles": (_i, [_vp, _i, _i64, _i, _vp, _vp, _vp]),
    "cl_channel_histogram": (_i, [_vp, _vp, _i64, _i, _i, _i, _d, _d, _vp, _vp, _vp]),
    "cl_de_trial": (_i, [_vp, _i, _i, _d, _d, _d, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cl_de_select": (_i, [_vp, _vp, _vp, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _vp]),
    "cl_quantize_8bit_workspace_bytes": (_sz, []),
    "cl_quantize_8bit": (_i, [_vp, _i64, _d, _vp, _vp, _vp, _sz, _vp]),
    "cl_pair_statistics_workspace_bytes": (_sz, [_i]),
    "cl_pair_statistics": (_i, [_vp, _vp, _vp, _vp, _d, C.POINTER(C.c_double), C.POINTER(C.c_double), _i64, _i,
                                _vp, _vp, _sz, _vp]),
}

_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (once) and return the CUDA library.  Raises if it is missing -- never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if build_if_missing:
            from . import build as _build
            _build.build()
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m camera_linearity_b200.build` "
                "(needs nvcc).  camera_linearity_b200 has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.cl_abi_version() != 1:
        raise RuntimeError("libcamlin_b200.so ABI version mismatch; rebuild the library")
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().cl_status_string(status)
        raise CamlinError(status, what, msg.decode() if msg else "?")


def launch_count() -> int:
    return int(load().cl_launch_count())
