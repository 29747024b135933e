"""ctypes binding of ``lib/libibs_b200.so`` (the C ABI declared in ``include/ibs_b200.h``).

PyTorch is used by the callers for device memory and streams only; the signatures here carry
plain pointers and sizes.  There is no CPU fallback: ``load()`` raises if the library has not been
built, and ``require_cuda()`` raises if no GPU is visible.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IBS_LIB") or os.path.join(HERE, "lib", "libibs_b200.so")      # IBS_LIB: tuning builds

_D = c_void_p      # device/host double*
_I = c_void_p      # int*

#: every symbol declared in include/ibs_b200.h with its ctypes signature
SIGNATURES = {
    "ibs_version": (c_int, []),
    "ibs_last_error": (c_char_p, []),
    "ibs_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "ibs_fp64_probe": (c_int, [c_int, _D, ctypes.c_longlong, POINTER(c_double), c_void_p]),
    "ibs_geometry_batch": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double,
                                   _D, c_int, c_int, _D, c_int, c_double, _D, _D, _D, _I, c_void_p]),
    "ibs_geometry_tangent_batch": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double,
                                           _D, c_int, c_int, _D, c_int, c_double, _D, _D, _D, _D, _D, _I, c_void_p]),
    "ibs_geometry_full_nfields": (c_int, []),
    "ibs_geometry_full": (c_int, [_D, _D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double, _D, c_int, _D, c_int,
                                  c_int, c_double, c_int, c_double, _D, _I, c_void_p]),
    "ibs_geometry_adjoint": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double, _D, _D, c_int, c_double,
                                     _D, _D, _D, _D, _D, _D, _D, _D, c_void_p]),
    "ibs_geometry_adjoint_scal": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double, _D, _D, c_int,
                                          c_double, _D, _D, _D, _D, _D, _D, _D, _D, _D, _D, c_void_p]),
    "ibs_solve_gcf_batch": (c_int, [_D, _D, _D, c_int, c_int, c_double, _D, _D, c_int, _D, _D, _D, _D, _I, c_void_p]),
    "ibs_solve_base_batch": (c_int, [_D, _D, _D, _I, c_int, c_int, c_int, c_double, _D, _D, c_int,
                                     _D, _D, _D, _D, _D, _D, _D, _I, c_void_p]),
    "ibs_adjoint_batch": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, _D, c_void_p]),
    "ibs_adjoint_sensitivities": (c_int, [_D, _D, _D, _D, c_int, c_int, _D, _D, _D, c_void_p]),
    "ibs_obj_w_grad_batch": (c_int, [_D, _D, _D, c_int, c_int, c_double, c_double, _D, _D, _D, _D, _D, _I, c_void_p]),
    "ibs_obj_w_grad_tangent_batch": (c_int, [_D, _D, _D, _D, _D, c_int, c_int, c_double, _D, _D, _D, _D, _D, _I, c_void_p]),
    "ibs_scan_argmax": (c_int, [_D, c_int, c_int, _D, _I, _D, c_void_p]),
    "ibs_refine_state_doubles": (c_int, []),
    "ibs_refine_init": (c_int, [_D, c_int, _D, _D, c_double, c_double, c_double, c_double, c_double, _D, _D, c_void_p]),
    "ibs_refine_step": (c_int, [_D, c_int, _D, _D, _I, c_double, c_double, c_int, c_double, _D, _D, _I, c_void_p]),
    "ibs_count_above_batch": (c_int, [_D, _D, _D, c_int, c_int, c_double, _D, _I, c_void_p]),
    "ibs_scan_solve_argmax": (c_int, [_D, _D, _D, c_int, c_int, c_int, c_int, c_double, _D, c_int, _D, _D, _D, _I, _D, _D, c_void_p]),
    "ibs_scan_host": (c_int, [_D, _D, _D, _D, _D, _D, _D, c_int, c_int, c_int, c_double, c_double,
                              _D, c_int, _D, c_int, _D, c_int, c_double, _D, _D, _I, _D, _D, _D, _I]),
}

_lib = None


class IbsError(RuntimeError):
    pass


def load(build_if_missing: bool = False):
    """Load the shared library (once) and attach the signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        if build_if_missing:
            from . import build as _build
            _build.build()
        else:
            raise IbsError(f"{LIB_PATH} is missing: run `python -m ideal_ballooning_solver_b200.build` "
                           "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().ibs_last_error()
        raise IbsError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise IbsError("no CUDA device visible: the ballooning engine has no CPU fallback")
