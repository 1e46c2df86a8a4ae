"""ctypes binding of csrc/libnnmpc.so (the C ABI declared in include/nnmpc.h).

The library is built in-tree by ``industrial_nnmpc_2021_b200.build``.  There is no CPU
fallback: ``lib()`` raises when the shared object is missing and every ``*_create`` call fails
when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libnnmpc.so")
if os.environ.get("NNMPC_LIB_PATH"):      # experimental build variants (build.py --out ...)
    LIB_PATH = os.environ["NNMPC_LIB_PATH"]

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
vp = C.c_void_p

# symbol -> (restype, argtypes); must list every function declared in include/nnmpc.h
SIGNATURES = {
    "nnmpc_version": (C.c_int, []),
    "nnmpc_last_error": (C.c_char_p, []),
    "nnmpc_launch_count": (C.c_longlong, []),
    "nnmpc_iteration_count": (C.c_longlong, []),
    "nnmpc_prof_enable": (C.c_int, [C.c_int]),
    "nnmpc_prof_read": (C.c_int, [c_double_p, c_double_p, C.POINTER(C.c_longlong), C.c_int]),
    "nnmpc_prof_read2": (C.c_int, [c_double_p, c_double_p, C.POINTER(C.c_longlong), C.c_int]),
    "nnmpc_prof_readn": (C.c_int, [C.c_int, c_double_p, c_double_p, C.POINTER(C.c_longlong), C.c_int]),
    "nnmpc_qp_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp,
                                  C.c_double, C.c_int]),
    "nnmpc_qp_create_ipm": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_int]),
    "nnmpc_qp_set_penalty": (C.c_int, [vp, vp]),
    "nnmpc_qp_destroy": (C.c_int, [vp]),
    "nnmpc_qp_solve": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, C.c_double, C.c_int, vp]),
    "nnmpc_qp_solve_host": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_int]),
    "nnmpc_ts_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                  vp, C.c_int]),
    "nnmpc_ts_set_output_bounds": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp]),
    "nnmpc_ts_create_reduced": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
                                + [vp] * 16 + [C.c_int]),
    "nnmpc_ts_destroy": (C.c_int, [vp]),
    "nnmpc_ts_solve": (C.c_int, [vp, C.c_int, vp, C.c_longlong, vp, C.c_longlong, vp, vp, vp, vp]),
    "nnmpc_ts_solve_host": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp]),
    "nnmpc_sim_create": (C.c_int, [C.POINTER(vp), vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int]),
    "nnmpc_sim_destroy": (C.c_int, [vp]),
    "nnmpc_sim_set_precision": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_set_slots": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_set_cadence": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_set_tail_rows": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_set_exact_gemm": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_set_capture": (C.c_int, [vp, vp, vp]),
    "nnmpc_sim_set_one_term_threshold": (C.c_int, [vp, C.c_double]),
    "nnmpc_sim_tile_stats": (C.c_int, [vp, C.POINTER(C.c_longlong)]),
    "nnmpc_sim_set_second_term_cadence": (C.c_int, [vp, C.c_int]),
    "nnmpc_sim_stats": (C.c_int, [vp, C.POINTER(C.c_longlong)]),
    "nnmpc_sim_active_stats": (C.c_int, [vp, C.POINTER(C.c_longlong)]),
    "nnmpc_sim_run": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_double,
                                C.c_int, C.c_int, vp]),
    "nnmpc_sim_solve_qps": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_int, vp]),
    "nnmpc_sim_run_host": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_double,
                                     C.c_int, C.c_int]),
    "nnmpc_mlp_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_int, c_int_p, C.POINTER(vp),
                                   C.POINTER(vp), C.c_int]),
    "nnmpc_mlp_destroy": (C.c_int, [vp]),
    "nnmpc_mlp_set_precision": (C.c_int, [vp, C.c_int]),
    "nnmpc_mlp_train_step": (C.c_int, [vp, C.c_longlong, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_double, C.c_double,
                                       C.c_longlong, C.c_int, c_double_p, vp]),
    "nnmpc_mlp_get_weights": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "nnmpc_mlp_forward": (C.c_int, [vp, C.c_longlong, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nnmpc_mlp_forward_host": (C.c_int, [vp, C.c_longlong, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nnmpc_online_create": (C.c_int, [C.POINTER(vp), vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp,
                                      vp, vp, vp, vp, vp, C.c_int]),
    "nnmpc_online_destroy": (C.c_int, [vp]),
    "nnmpc_online_run": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                   vp, C.c_double, C.c_int, vp]),
    "nnmpc_lp_gemm_test": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, vp, C.c_double, vp, C.c_int, vp]),
    "nnmpc_lp_pass_probe": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "nnmpc_oz_gemm_test": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    "nnmpc_exact_apply_test": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp,
                                         vp, vp, vp, vp, vp, vp]),
    "nnmpc_lp_step_test": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, vp, C.c_double]
                           + [vp] * 6 + [vp, C.c_int, C.c_int] + [vp] * 21),
    "nnmpc_gemm_tn": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, C.c_longlong, vp, C.c_longlong, vp, C.c_longlong,
                                vp, vp]),
}

NNMPC_WARN_MAXITER = 1      # warnings are a bit mask (include/nnmpc.h)
NNMPC_WARN_TARGET = 2
_lib = None


class NnmpcError(RuntimeError):
    pass


def lib():
    """Load libnnmpc.so (once).  Raises if it has not been built - there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NnmpcError(
            f"{LIB_PATH} is missing: build it with `python -m industrial_nnmpc_2021_b200.build` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return _lib


def check(rc, what=""):
    """Raise on a negative status and on a target-selector solve that missed its optimum (a wrong
    target would silently corrupt everything built on it); return True when some regulator QP
    reached max_iter (its kkt entry tells which)."""
    if rc < 0:
        msg = lib().nnmpc_last_error().decode(errors="replace")
        raise NnmpcError(f"{what} failed (status {rc}): {msg}")
    if rc & NNMPC_WARN_TARGET:
        raise NnmpcError(f"{what}: a target-selector solve did not reach its optimum (active-set stall or "
                         "non-finite data)")
    return bool(rc & NNMPC_WARN_MAXITER)


def host(a):
    """C-contiguous float64 view/copy of a host array."""
    return np.ascontiguousarray(a, dtype=np.float64)


def hptr(a):
    """void* of a contiguous NumPy array (or None)."""
    return None if a is None else a.ctypes.data_as(vp)


def dptr(t, dtype=None, device=None):
    """void* of a contiguous CUDA torch tensor (or None).  The C ABI reinterprets the bytes, so the
    element type (default float64) and, when given, the device index are checked here."""
    if t is None:
        return None
    import torch
    want = torch.float64 if dtype is None else dtype
    if not t.is_cuda or not t.is_contiguous():
        raise NnmpcError("expected a contiguous CUDA tensor")
    if t.dtype != want:
        raise NnmpcError(f"expected a {want} tensor, got {t.dtype}")
    if device is not None and t.device.index != device:
        raise NnmpcError(f"tensor lives on cuda:{t.device.index}, the handle on cuda:{device}")
    return vp(t.data_ptr())


def dptr_i32(t, device=None):
    import torch
    return dptr(t, torch.int32, device)


def prof_enable(on=True):
    """Switch the live CUDA-event timing of the iteration GEMM on/off (bench.py roofline)."""
    check(lib().nnmpc_prof_enable(int(bool(on))), "nnmpc_prof_enable")


def prof_read(reset=True):
    """(device ms, algorithmic flops, launches) of the iteration GEMM since the last reset."""
    ms, fl, n = C.c_double(), C.c_double(), C.c_longlong()
    check(lib().nnmpc_prof_read(C.byref(ms), C.byref(fl), C.byref(n), int(bool(reset))), "nnmpc_prof_read")
    return ms.value, fl.value, n.value


def prof_read2(reset=True):
    """Two-channel form: [(ms, flops, launches) of the iteration passes, (...) of the FP64 anchor /
    exact-check GEMMs of the mixed-precision mode]."""
    ms, fl, n = (C.c_double * 2)(), (C.c_double * 2)(), (C.c_longlong * 2)()
    check(lib().nnmpc_prof_read2(ms, fl, n, int(bool(reset))), "nnmpc_prof_read2")
    return [(ms[i], fl[i], n[i]) for i in range(2)]


def prof_readn(nchan=4, reset=True):
    """[(ms, flops, launches)] per channel: 0 iteration passes, 1 exact anchors / KKT checks, 2 FP64 tail
    iterations, 3 the rest of a full engine loop."""
    ms, fl, n = (C.c_double * nchan)(), (C.c_double * nchan)(), (C.c_longlong * nchan)()
    check(lib().nnmpc_prof_readn(nchan, ms, fl, n, int(bool(reset))), "nnmpc_prof_readn")
    return [(ms[i], fl[i], n[i]) for i in range(nchan)]


PRECISION = {"f64": 0, "mixed": 1}


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on the handle's device."""
    import torch
    return vp(torch.cuda.current_stream(device).cuda_stream)
