"""ctypes binding of include/marlpde_b200.h (the C-ABI shared library built from csrc/).

The library is the product; this module only loads it and mirrors its structs.  There is no
fallback: if the library is missing, or the box has no CUDA device, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MARLPDE_B200_LIB") or os.path.join(_HERE, "libmarlpde_b200.so")

NFIELDS = 5
NEVENTS = 7
STATUS_FINISHED, STATUS_STEP_TOO_SMALL, STATUS_NONFINITE, STATUS_STEP_BUDGET = 0, -1, -2, 1
FLAG_EVENTS = 1
FLAG_QUEUE_LOCKS = 2
FLAG_VAR_DPHI = 4
FLAG_QUEUE_TAIL = 8
FLAG_JAC_FD = 16
MODEL_VAR_DPHI = 1


class ColumnParams(C.Structure):
    _fields_ = [("bc_top", C.c_double * 5), ("dx", C.c_double), ("inv_dx", C.c_double),
                ("inv_dx2", C.c_double), ("delta_x", C.c_double), ("presum", C.c_double),
                ("rhorat", C.c_double), ("Da", C.c_double), ("lambda_", C.c_double),
                ("dCa", C.c_double), ("dCO3", C.c_double), ("delta", C.c_double), ("KRat", C.c_double),
                ("nu1", C.c_double), ("nu2", C.c_double), ("m1", C.c_double), ("m2", C.c_double),
                ("n1", C.c_double), ("n2", C.c_double), ("dPhi_fixed", C.c_double),
                ("Peclet_min", C.c_double), ("Peclet_max", C.c_double), ("FV_switch", C.c_int32),
                ("mask_lo", C.c_int32), ("mask_hi", C.c_int32), ("model_flags", C.c_int32),
                ("auxcon", C.c_double)]


class RK45Options(C.Structure):
    _fields_ = [("t_bound", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
                ("max_step", C.c_double), ("max_steps", C.c_int64), ("n_eval", C.c_int32),
                ("event_capacity", C.c_int32), ("flags", C.c_int32), ("quantum", C.c_int32)]


class ColumnState(C.Structure):
    _fields_ = [("t", C.c_double), ("h_abs", C.c_double), ("n_accepted", C.c_int64),
                ("n_rejected", C.c_int64), ("nfev", C.c_int64), ("status", C.c_int32),
                ("next_eval", C.c_int32)]


class DeviceInfo(C.Structure):
    _fields_ = [("name", C.c_char * 128), ("sm_count", C.c_int32), ("cc_major", C.c_int32),
                ("cc_minor", C.c_int32), ("max_smem_per_block", C.c_int32), ("total_mem", C.c_int64)]


# numpy views of the structs (same memory layout; used for vectorised host-side set-up)
PARAMS_DTYPE = np.dtype([("bc_top", "<f8", (5,)), ("dx", "<f8"), ("inv_dx", "<f8"), ("inv_dx2", "<f8"),
                         ("delta_x", "<f8"), ("presum", "<f8"), ("rhorat", "<f8"), ("Da", "<f8"),
                         ("lambda_", "<f8"), ("dCa", "<f8"), ("dCO3", "<f8"), ("delta", "<f8"),
                         ("KRat", "<f8"), ("nu1", "<f8"), ("nu2", "<f8"), ("m1", "<f8"), ("m2", "<f8"),
                         ("n1", "<f8"), ("n2", "<f8"), ("dPhi_fixed", "<f8"), ("Peclet_min", "<f8"),
                         ("Peclet_max", "<f8"), ("FV_switch", "<i4"), ("mask_lo", "<i4"),
                         ("mask_hi", "<i4"), ("model_flags", "<i4"), ("auxcon", "<f8")])
STATE_DTYPE = np.dtype([("t", "<f8"), ("h_abs", "<f8"), ("n_accepted", "<i8"), ("n_rejected", "<i8"),
                        ("nfev", "<i8"), ("status", "<i4"), ("next_eval", "<i4")])
assert PARAMS_DTYPE.itemsize == C.sizeof(ColumnParams)
assert STATE_DTYPE.itemsize == C.sizeof(ColumnState)

# every symbol include/marlpde_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "marlpde_abi_version": (C.c_int, []),
    "marlpde_struct_size": (C.c_int, [C.c_int]),
    "marlpde_last_error": (C.c_char_p, []),
    "marlpde_device_count": (C.c_int, []),
    "marlpde_get_device_info": (C.c_int, [C.c_int, C.POINTER(DeviceInfo)]),
    "marlpde_release_cached_memory": (C.c_int, []),
    "marlpde_rk45_max_cells": (C.c_int, []),
    "marlpde_rk45_columns_per_cta": (C.c_int, [C.c_int]),
    "marlpde_rhs_batch_dev": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P]),
    "marlpde_rhs_batch": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int]),
    "marlpde_rk45_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                             _P, _P, _P, _P, _P, _P]),
    "marlpde_rk45_integrate_async": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options), _P, _P, _P, _P,
                                               C.c_int, _P]),
    "marlpde_rk45_stream_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "marlpde_rk45_stream_integrate_events_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                                           _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "marlpde_rk45_stream_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                                    _P, _P, _P, C.c_size_t, _P]),
    "marlpde_radau_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "marlpde_radau_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                              _P, _P, _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "marlpde_radau_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                          _P, _P, _P, _P, _P, C.c_int]),
    "marlpde_radau_integrate_async": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                                _P, _P, _P, _P, _P, C.c_int, _P]),
    "marlpde_bdf_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "marlpde_bdf_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                            _P, _P, _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "marlpde_bdf_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                        _P, _P, _P, _P, _P, C.c_int]),
    "marlpde_bdf_integrate_async": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                              _P, _P, _P, _P, _P, C.c_int, _P]),
    "marlpde_bdf_sens_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "marlpde_bdf_sens_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                                 _P, _P, _P, _P, _P, _P, C.c_size_t, _P, C.c_int,
                                                 _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "marlpde_bdf_sens_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                             _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int]),
    "marlpde_rk23_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "marlpde_rk23_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                             _P, _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "marlpde_rk23_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                         _P, _P, _P, _P, C.c_int]),
    "marlpde_rk23_integrate_async": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                               _P, _P, _P, _P, C.c_int, _P]),
    "marlpde_dop853_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "marlpde_dop853_integrate_dev": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                               _P, _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "marlpde_dop853_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                           _P, _P, _P, _P, C.c_int]),
    "marlpde_dop853_integrate_async": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                                 _P, _P, _P, _P, C.c_int, _P]),
    "marlpde_probe_jacobian":(C.c_int, [_P, _P, C.c_int, _P, C.c_int]),
    "marlpde_probe_math": (C.c_int, [C.c_int, _P, C.c_int, _P, C.c_int]),
    "marlpde_probe_fp64_peak": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "marlpde_rk45_integrate": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.POINTER(RK45Options),
                                         _P, _P, _P, _P, C.c_int]),
}


class MarlpdeError(RuntimeError):
    pass


_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once). Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MarlpdeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). The CUDA library is the only implementation; there is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.marlpde_abi_version() != 2:
            raise MarlpdeError("ABI version mismatch between _cabi.py and libmarlpde_b200.so")
        for which, struct in enumerate((ColumnParams, RK45Options, ColumnState, DeviceInfo)):
            if handle.marlpde_struct_size(which) != C.sizeof(struct):
                raise MarlpdeError(f"struct layout mismatch for {struct.__name__}")
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().marlpde_last_error().decode("utf-8", "replace")
        raise MarlpdeError(f"marlpde_b200 error {rc}: {msg}")


def ptr(a) -> int | None:
    """Address of a C-contiguous numpy array / torch tensor (None -> NULL)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return a.ctypes.data
    return a.data_ptr()  # torch tensor
