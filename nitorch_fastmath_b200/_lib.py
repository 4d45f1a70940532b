"""ctypes binding of ``libnfm_sm100a.so`` (C ABI: ``include/nfm.h``).

The library is the product: there is NO fallback.  If it is missing, or no
CUDA device is present, every operation raises -- it never silently computes
with torch or on the CPU.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_int, c_int64, c_size_t, c_uint64, c_void_p

LIB_NAME = "libnfm_sm100a.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

F32, F64 = 0, 1
LAYOUT_SCALED_IDENTITY, LAYOUT_DIAG, LAYOUT_SYM, LAYOUT_FULL = 0, 1, 2, 3
ALGO_AUTO, ALGO_LDL, ALGO_LU, ALGO_WARP = 0, 1, 2, 3
MAX_N = 10

_P, _I, _L = c_void_p, c_int, c_int64


class NfmOperand(ctypes.Structure):
    """``nfm_operand`` of include/nfm.h: pointer, batch stride, element stride (in elements)."""
    _fields_ = [("ptr", c_void_p), ("batch_stride", c_int64), ("elem_stride", c_int64)]


_O = ctypes.POINTER(NfmOperand)

# name -> (restype, argtypes); mirrors include/nfm.h declaration by declaration
SIGNATURES = {
    "nfm_version": (c_int, []),
    "nfm_last_error_string": (ctypes.c_char_p, []),
    "nfm_launch_count": (c_uint64, []),
    "nfm_last_path_was_tma": (c_int, []),
    "nfm_last_launch_shape": (c_int, [ctypes.POINTER(c_int64)]),
    "nfm_sym_matvec": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _I, _P, _L, _P]),
    "nfm_sym_solve": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_invert": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_matvec_ex": (c_int, [_I, _I, _I, _L, _O, _O, _O, _I, _O, _P]),
    "nfm_sym_solve_ex": (c_int, [_I, _I, _I, _I, _L, _O, _O, _O, _O, _P]),
    "nfm_sym_invert_ex": (c_int, [_I, _I, _I, _I, _L, _O, _O, _P]),
    "nfm_batch_inv": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_det": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_solve": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_rsolve": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_matvec": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_det": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_to_full": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_outer": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_matmul": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_solve_update": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, ctypes.c_double, ctypes.c_double, _P, _L, _P]),
    "nfm_sym_matmul_solve": (c_int, [_I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_solve_update_reg": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P, _L, ctypes.c_double, ctypes.c_double, _P, _L, _P]),
    "nfm_sym_outer2": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _I, _P, _L, _P]),
    "nfm_sym_invert_backward": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_det_backward": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_matmul_backward": (c_int, [_I, _I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_outer_backward": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_sym_to_full_backward": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_det_backward": (c_int, [_I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_inv_backward": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_outer": (c_int, [_I, _I, _I, _I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_tsolve": (c_int, [_I, _I, _I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_batch_tmatvec": (c_int, [_I, _I, _I, _L, _P, _L, _P, _L, _P, _L, _P]),
    "nfm_host_workspace_bytes": (c_size_t, [_I, _L, _I, _I, _I]),
    "nfm_sym_solve_host": (c_int, [_I, _I, _I, _L, _P, _P, _P, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
    "nfm_sym_invert_host": (c_int, [_I, _I, _I, _I, _L, _P, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
    "nfm_sym_matvec_host": (c_int, [_I, _I, _L, _P, _P, _P, _I, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
    "nfm_batch_inv_host": (c_int, [_I, _I, _I, _I, _L, _P, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
    "nfm_batch_det_host": (c_int, [_I, _I, _L, _P, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
    "nfm_batch_solve_host": (c_int, [_I, _I, _I, _I, _L, _P, _P, _P, _P, c_size_t, _L, _I, ctypes.POINTER(c_void_p)]),
}

_lib = None


class NfmError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NfmError(
                f"{LIB_PATH} not found: build it with `make -C nitorch_fastmath_b200/csrc -j8` "
                "(or __graft_entry__.build()).  There is no CPU / torch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().nfm_last_error_string().decode("utf-8", "replace")
        raise NfmError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().nfm_launch_count())


LAUNCH_FIELDS = ("kind", "threads", "mpt", "stages", "warps", "seg", "grid", "tiles")


def last_launch_shape() -> dict:
    """The bulk launch of the last call on this thread (``nfm_last_launch_shape``)."""
    buf = (c_int64 * 8)()
    check(load().nfm_last_launch_shape(buf), "nfm_last_launch_shape")
    return dict(zip(LAUNCH_FIELDS, (int(v) for v in buf)))
