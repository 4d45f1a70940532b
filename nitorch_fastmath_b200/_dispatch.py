"""Host-side plumbing between torch tensors and the C ABI.

torch is used for allocation, broadcasting metadata and the current stream
only.  Every operand is handed to the library as (device pointer, batch
stride, element stride), all in elements: its batch dims must collapse to one
stride -- 0 for a fully broadcast operand, ``record length`` for a dense one,
anything else takes the library's strided kernel.  A 1-D record whose elements
are not adjacent (a channel-first field viewed coefficient-last) is passed
with its element stride; 2-D records must be contiguous.  Operands whose
batch dims do not collapse are materialised with ``.contiguous()`` (one extra
pass; documented in DESIGN.md).
"""
from __future__ import annotations

import itertools
import math
from typing import Optional, Sequence, Tuple

import torch

from . import _lib

_DTYPE_CODE = {torch.float32: _lib.F32, torch.float64: _lib.F64}


def dtype_code(dtype: torch.dtype) -> int:
    try:
        return _DTYPE_CODE[dtype]
    except KeyError:
        raise TypeError(f"nitorch_fastmath_b200 supports float32 and float64, got {dtype}") from None


def compute_dtype(*tensors, dtype: Optional[torch.dtype] = None) -> torch.dtype:
    if dtype is None:
        dtype = tensors[0].dtype
        for t in tensors[1:]:
            dtype = torch.promote_types(dtype, t.dtype)
    if dtype not in _DTYPE_CODE:
        if dtype.is_floating_point:      # half / bfloat16 inputs compute in float32
            dtype = torch.float32
        else:
            raise TypeError(f"unsupported dtype {dtype}")
    return dtype


def common_device(*tensors) -> torch.device:
    dev = tensors[0].device
    for t in tensors[1:]:
        if t.device != dev:
            raise RuntimeError(f"operands live on different devices: {dev} and {t.device}")
    return dev


def check_order(n: int) -> int:
    if not 1 <= n <= _lib.MAX_N:
        raise ValueError(f"matrix order {n} is outside the supported range 1..{_lib.MAX_N}")
    return n


def _record_contiguous(t: torch.Tensor, rec_ndim: int) -> bool:
    expect = 1
    for d in range(t.dim() - 1, t.dim() - 1 - rec_ndim, -1):
        if t.shape[d] != 1 and t.stride(d) != expect:
            return False
        expect *= t.shape[d]
    return True


def _collapse(shape: Sequence[int], strides: Sequence[int]) -> Optional[int]:
    """Single stride that walks ``shape`` in row-major order, or None."""
    dims = [(n, s) for n, s in zip(shape, strides) if n != 1]
    if not dims:
        return None  # single element: any stride works
    for (n0, s0), (n1, s1) in zip(dims[:-1], dims[1:]):
        if s0 != s1 * n1:
            return -1
    return dims[-1][1]


class Operand:
    """(pointer, batch stride, element stride) view of a tensor; keeps the storage alive."""
    __slots__ = ("tensor", "ptr", "stride", "estride")

    def __init__(self, tensor: torch.Tensor, stride: int, estride: int = 1):
        self.tensor = tensor
        self.ptr = tensor.data_ptr()
        self.stride = stride
        self.estride = estride

    def c_struct(self) -> "_lib.NfmOperand":
        return _lib.NfmOperand(self.ptr, self.stride, self.estride)


def as_operand(t: torch.Tensor, batch_shape: Tuple[int, ...], rec_ndim: int, dtype: torch.dtype,
               allow_estride: bool = False) -> Operand:
    """Broadcast ``t``'s batch dims to ``batch_shape`` and express it as one
    batch stride.  With ``allow_estride`` a 1-D record whose elements are not
    adjacent (coefficient-first storage viewed coefficient-last) is passed as
    is, with its element stride, instead of being copied."""
    if t.dtype != dtype:
        t = t.to(dtype)
    rec_shape = tuple(t.shape[t.dim() - rec_ndim:]) if rec_ndim else ()
    rec_len = math.prod(rec_shape)
    estride = 1
    nb = len(batch_shape)
    if not _record_contiguous(t, rec_ndim):
        full = t.expand(*batch_shape, *rec_shape)
        bstride = _collapse(full.shape[:nb], full.stride()[:nb])
        if allow_estride and rec_ndim == 1 and t.stride(-1) > 0 and (bstride is None or bstride > 0):
            estride = t.stride(-1)          # strided record, collapsible non-broadcast batch: no copy
        else:
            t = t.contiguous()
    full = t.expand(*batch_shape, *rec_shape)
    stride = _collapse(full.shape[:nb], full.stride()[:nb])
    if stride is None:
        stride = rec_len if estride == 1 else 0
    elif stride < 0:
        full = full.contiguous()
        stride, estride = rec_len, 1
    return Operand(full, stride, estride)


def check_out_shape(out: Optional[torch.Tensor], shape: Sequence[int]) -> None:
    """``out`` must have exactly the result's shape: the host pipelines write ``batch x record``
    elements through its pointer, and ``copy_`` would broadcast into a larger tensor."""
    if out is not None and tuple(out.shape) != tuple(shape):
        raise RuntimeError(f"out has shape {tuple(out.shape)}, expected {tuple(shape)}")


def out_operand(out: Optional[torch.Tensor], shape: Tuple[int, ...], rec_ndim: int, dtype: torch.dtype,
                device: torch.device, allow_estride: bool = False):
    """Returns (operand to write into, tensor to return, needs_copy_back)."""
    if out is None:
        res = torch.empty(shape, dtype=dtype, device=device)
        rec_len = math.prod(shape[len(shape) - rec_ndim:]) if rec_ndim else 1
        return Operand(res, rec_len), res, False
    check_out_shape(out, shape)
    if out.device != device:
        raise RuntimeError("out lives on a different device")
    nb = len(shape) - rec_ndim
    estride = 1
    ok = out.dtype == dtype
    if ok and not _record_contiguous(out, rec_ndim):
        if allow_estride and rec_ndim == 1 and out.stride(-1) > 0:
            estride = out.stride(-1)
        else:
            ok = False
    stride = _collapse(out.shape[:nb], out.stride()[:nb]) if ok else -1
    rec_len = math.prod(shape[nb:]) if rec_ndim else 1
    if stride is None:
        stride = rec_len if estride == 1 else 0
    if not ok or stride < 0 or (stride == 0 and math.prod(shape[:nb]) > 1):
        tmp = torch.empty(shape, dtype=dtype, device=device)
        return Operand(tmp, rec_len), out, True
    return Operand(out, stride, estride), out, False


def outer_split(batch_shape: Tuple[int, ...], operands: Sequence[Tuple[Optional[torch.Tensor], int]],
                max_outer: int = 512) -> int:
    """Partially broadcast operands (e.g. one Hessian field ``(1, X, Y, Z, NN)`` for a batch of
    gradient fields ``(B, X, Y, Z, N)``) do not collapse to one batch stride.  Instead of
    materialising them, the leading ``s`` batch dims can be looped over: returns the smallest
    ``s > 0`` such that every operand, expanded to ``batch_shape``, collapses over dims ``[s:]``
    -- or 0 when no split is needed, none exists, or it would take more than ``max_outer`` launches."""
    nb = len(batch_shape)

    def collapses(s: int) -> bool:
        for t, rec_ndim in operands:
            if t is None:
                continue
            rec_shape = tuple(t.shape[t.dim() - rec_ndim:]) if rec_ndim else ()
            full = t.expand(*batch_shape, *rec_shape)
            c = _collapse(full.shape[s:nb], full.stride()[s:nb])
            if c is not None and c < 0:
                return False
        return True

    if nb < 2 or collapses(0):
        return 0
    for s in range(1, nb):
        if math.prod(batch_shape[:s]) > max_outer:
            return 0
        if collapses(s):
            return s
    return 0


def outer_views(t: Optional[torch.Tensor], batch_shape: Tuple[int, ...], rec_ndim: int, idx: Tuple[int, ...]):
    """The slice ``idx`` (over the leading batch dims) of ``t`` expanded to ``batch_shape``: a view."""
    if t is None:
        return None
    rec_shape = tuple(t.shape[t.dim() - rec_ndim:]) if rec_ndim else ()
    return t.expand(*batch_shape, *rec_shape)[idx]


def outer_loop(batch: Tuple[int, ...], operands: Sequence[Tuple[Optional[torch.Tensor], int]],
               out: Optional[torch.Tensor], rec: Tuple[int, ...], dtype: torch.dtype, device: torch.device,
               call) -> Optional[torch.Tensor]:
    """Partially broadcast operands (see ``outer_split``): ``call(*operand views, out view)`` once per
    index of the leading batch dims, on views, so nothing is materialised and each call sees dense or
    fully broadcast operands.  Returns ``out`` (or a new ``dtype`` tensor) filled, or None when no
    split applies and the caller launches once."""
    split = outer_split(batch, operands) if batch_count(batch) > 0 else 0
    if not split:
        return None
    shape = (*batch, *rec)
    full = out if (out is not None and out.dtype == dtype and tuple(out.shape) == shape) else \
        torch.empty(shape, dtype=dtype, device=device)
    for idx in itertools.product(*[range(k) for k in batch[:split]]):
        call(*[outer_views(t, batch, nd, idx) for t, nd in operands], full[idx])
    if out is not None and full is not out:
        out.copy_(full)
        return out
    return full


def batch_count(batch_shape: Sequence[int]) -> int:
    return math.prod(batch_shape)


def launch(fn_name: str, head: Sequence, batch: Tuple[int, ...],
           operands: Sequence[Tuple[Optional[torch.Tensor], int]], tail: Sequence = (), *,
           rec: Tuple[int, ...], out: Optional[torch.Tensor] = None, dtype: torch.dtype, device: torch.device,
           struct: bool = False, skip_empty: bool = False, what: Optional[str] = None) -> torch.Tensor:
    """Run the device entry ``fn_name(dtype code, *head, nb, *operands, *tail, out, stream)`` over
    ``batch`` on ``device`` and return its ``(*batch, *rec)`` result (``out`` when given).

    Each ``(tensor, rec_ndim)`` operand is broadcast to ``batch`` and passed as (pointer, batch
    stride), an absent one as (NULL, 0).  With ``struct`` the ``fn_name + "_ex"`` entry is called
    with ``nfm_operand`` pointers, which also carry an element stride, so strided 1-D records are
    passed without a copy; an absent operand is a NULL struct.  An ``out`` the library cannot write
    through (another dtype, batch dims that do not collapse) is written through a temporary and
    copied back.  The call is skipped when the batch is empty, or with ``skip_empty`` when the result
    is; errors are reported as ``what`` (default ``fn_name``)."""
    o, res, copy_back = out_operand(out, batch + rec, len(rec), dtype, device, struct)
    nb = math.prod(batch)
    if nb > 0 and not (skip_empty and res.numel() == 0):
        # ``ops`` keeps every Operand, and with it any converted or materialised copy, alive until
        # the call has been enqueued: the pointers below would otherwise dangle
        ops = [None if t is None else as_operand(t, batch, nd, dtype, struct) for t, nd in operands]
        if struct:
            args = [None if x is None else x.c_struct() for x in ops] + [*tail, o.c_struct()]
        else:
            args = [v for x in ops for v in ((None, 0) if x is None else (x.ptr, x.stride))] + [*tail, o.ptr, o.stride]
        fn = getattr(_lib.load(), fn_name + "_ex" if struct else fn_name)
        with device_of(device):
            rc = fn(dtype_code(dtype), *head, nb, *args, current_stream_ptr(device))
        _lib.check(rc, what or fn_name)
    if copy_back:
        res.copy_(o.tensor)
    return res


def current_stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def packed_order(length: int) -> int:
    """N from N(N+1)/2 (reference: _impl/sym.py:37)."""
    n = int((math.sqrt(1 + 8 * length) - 1) // 2)
    if n * (n + 1) // 2 != length:
        raise ValueError(f"{length} is not a packed-symmetric length N(N+1)/2")
    return n


def detect_layout(nn: int, n: int) -> int:
    """Compact layout from the two trailing sizes (reference sym.py:16-24)."""
    if nn == n * (n + 1) // 2:
        return _lib.LAYOUT_SYM      # also covers n == 1 where all four coincide
    if nn == 1:
        return _lib.LAYOUT_SCALED_IDENTITY
    if nn == n:
        return _lib.LAYOUT_DIAG
    if nn == n * n:
        return _lib.LAYOUT_FULL
    raise ValueError(f"matrix with {nn} coefficients does not match a vector of length {n}: "
                     f"expected 1, {n}, {n * (n + 1) // 2} or {n * n}")


# --------------------------------------------------------------------------
# fast path of the Python layer: dense CUDA operands with identical batch dims
# (the common case) skip the broadcasting / collapsing machinery above
# --------------------------------------------------------------------------

def plain_cuda(ref: torch.Tensor, *others: Optional[torch.Tensor]) -> bool:
    """All tensors are contiguous CUDA tensors on ref's device with ref's dtype
    (float32 / float64) and ref's batch dims (all dims but the last)."""
    if ref.device.type != "cuda" or ref.dtype not in _DTYPE_CODE or not ref.is_contiguous():
        return False
    lead = ref.shape[:-1]
    for t in others:
        if t is None:
            continue
        if t.device != ref.device or t.dtype != ref.dtype or not t.is_contiguous() or t.shape[:-1] != lead:
            return False
    return True


def empty_like_phased(ref: torch.Tensor, shape=None) -> torch.Tensor:
    """``torch.empty`` with ``ref``'s dtype / device whose address has the same offset from a
    16-byte boundary as ``ref``'s.  A dense view that starts inside its storage (``field[1:]``)
    is not 16-byte aligned; the library can still put it on the TMA path by peeling off a few
    leading matrices -- but only if the output, which has records of the same length, is out of
    phase by the same amount."""
    shape = tuple(ref.shape) if shape is None else tuple(shape)
    off = (ref.data_ptr() % 16) // ref.element_size()
    if off == 0:
        return torch.empty(shape, dtype=ref.dtype, device=ref.device)
    buf = torch.empty(math.prod(shape) + off, dtype=ref.dtype, device=ref.device)
    return buf[off:].view(shape)


class device_of:
    """Make ``dev`` current for the duration of a launch -- without touching the
    CUDA context when it already is (the usual case)."""
    __slots__ = ("_ctx",)

    def __init__(self, dev: torch.device):
        self._ctx = None if dev.index is None or dev.index == torch.cuda.current_device() else torch.cuda.device(dev)

    def __enter__(self):
        if self._ctx is not None:
            self._ctx.__enter__()

    def __exit__(self, *exc):
        if self._ctx is not None:
            self._ctx.__exit__(*exc)
