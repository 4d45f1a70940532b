"""Drop-in for ``nitorch_fastmath.batched`` (reference: nitorch_fastmath/batched.py,
nitorch_fastmath/_impl/batched.py): determinant, inverse and matrix-vector
product for large batches of small dense matrices, on hand-written sm_100a
kernels (orders 1..10; the reference's TorchScript closed forms stop at 3).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor

from . import _autograd as A
from . import _dispatch as D
from . import _host, _lib

__all__ = ['batchmatvec', 'batchdet', 'batchinv']


def _square_order(a: Tensor) -> int:
    if a.dim() < 2 or a.shape[-1] != a.shape[-2]:
        raise ValueError(f"expected (..., n, n) matrices, got {tuple(a.shape)}")
    n = a.shape[-1]
    if not 1 <= n <= _lib.MAX_N:
        raise ValueError(f"matrix order {n} is outside the supported range 1..{_lib.MAX_N}")
    return n


def _upload(*tensors):
    dev = _host.offload_device()
    return [t.to(dev, non_blocking=True) for t in tensors]


def _plain_host(*tensors) -> bool:
    """Contiguous float32 / float64 CPU tensors of one dtype: streamed through the GPU in
    chunks (nfm_batch_*_host); anything else is uploaded whole."""
    dt = tensors[0].dtype
    return dt in D._DTYPE_CODE and all(t.device.type == "cpu" and t.is_contiguous() and t.dtype == dt for t in tensors)


def batchdet(a: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    """Batched determinant of small matrices.

    Reference: _impl/batched.py:35-63 (closed forms det2/det3 :22-32; LU above).
    Differentiable (``nfm_batch_det_backward``): exact cofactors for n <= 3, also for
    singular matrices; above, g det(A) A^-T, which is not finite for a singular matrix.

    Parameters
    ----------
    a : (..., n, n) tensor

    Returns
    -------
    d : (...) tensor
    """
    if getattr(a, "requires_grad", False) and torch.is_grad_enabled():
        return A.batchdet(a, out)
    return _batchdet(a, out=out)


def _batchdet(a: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    a = torch.as_tensor(a)
    if a.device.type != "cuda":
        n = _square_order(a)
        nb = a.numel() // (n * n)
        D.check_out_shape(out, a.shape[:-2])
        if _plain_host(a) and nb > 0 and (out is None or _plain_host(a, out)):
            code = D.dtype_code(a.dtype)
            res = out if out is not None else torch.empty(a.shape[:-2], dtype=a.dtype, pin_memory=True)
            _host.run_host("nfm_batch_det_host", code, a.dtype, n * n, 1, nb,
                           lambda fn, ws, wsb, chunk, nbuf, streams: fn(code, n, nb, a.data_ptr(), res.data_ptr(), ws, wsb,
                                                                         chunk, nbuf, streams))
            return res
        r = batchdet(*_upload(a))
        if out is not None:
            out.copy_(r)
            return out
        return r.cpu()
    n = _square_order(a)
    cdt = D.compute_dtype(a)
    batch = tuple(a.shape[:-2])
    nb = D.batch_count(batch)
    o, res, copy_back = D.out_operand(out, batch, 0, cdt, a.device)
    if nb > 0:
        m = D.as_operand(a, batch, 2, cdt)
        with D.device_of(a.device):
            rc = _lib.load().nfm_batch_det(D.dtype_code(cdt), n, nb, m.ptr, m.stride, o.ptr, o.stride,
                                           D.current_stream_ptr(a.device))
        _lib.check(rc, "nfm_batch_det")
    if copy_back:
        res.copy_(o.tensor)
    return res


def batchinv(a: Tensor, *, method: str = 'auto', regularise: bool = True, out: Optional[Tensor] = None) -> Tensor:
    """Batched inversion of small matrices.

    Reference: _impl/batched.py:101-130.  Orders 2 and 3 use the reference's
    closed forms including its determinant shift ``det += (max|a|-min|a|)*1e-12``
    (:74-76, :94-96; ``regularise=False`` drops it); larger orders use
    Gauss-Jordan with partial pivoting in registers (the reference calls
    LAPACK there).  ``method='chol'`` inverts SPD matrices through LDL^T.

    Parameters
    ----------
    a : (..., n, n) tensor

    Returns
    -------
    a : (..., n, n) tensor

    Differentiable (``nfm_batch_inv_backward``); for orders 2 and 3 the determinant shift of
    ``regularise`` is treated as a constant.
    """
    if getattr(a, "requires_grad", False) and torch.is_grad_enabled():
        return A.batchinv(a, method, regularise, out)
    return _batchinv(a, method=method, regularise=regularise, out=out)


def _batchinv(a: Tensor, *, method: str = 'auto', regularise: bool = True, out: Optional[Tensor] = None) -> Tensor:
    a = torch.as_tensor(a)
    kind = method.lower()
    algo = {'auto': _lib.ALGO_AUTO, 'lu': _lib.ALGO_LU, 'chol': _lib.ALGO_LDL, 'ldl': _lib.ALGO_LDL}.get(kind)
    if algo is None:
        raise ValueError(f"unknown method {method!r}")
    if a.device.type != "cuda":
        n = _square_order(a)
        nb = a.numel() // (n * n)
        D.check_out_shape(out, a.shape)
        if _plain_host(a) and nb > 0 and (out is None or _plain_host(a, out)):
            code = D.dtype_code(a.dtype)
            res = out if out is not None else torch.empty(a.shape, dtype=a.dtype, pin_memory=True)
            _host.run_host("nfm_batch_inv_host", code, a.dtype, n * n, n * n, nb,
                           lambda fn, ws, wsb, chunk, nbuf, streams: fn(code, n, algo, int(bool(regularise)), nb, a.data_ptr(),
                                                                         res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        r = batchinv(*_upload(a), method=method, regularise=regularise)
        if out is not None:
            out.copy_(r)
            return out
        return r.cpu()
    n = _square_order(a)
    cdt = D.compute_dtype(a)
    batch = tuple(a.shape[:-2])
    nb = D.batch_count(batch)
    o, res, copy_back = D.out_operand(out, (*batch, n, n), 2, cdt, a.device)
    if nb > 0:
        m = D.as_operand(a, batch, 2, cdt)
        with D.device_of(a.device):
            rc = _lib.load().nfm_batch_inv(D.dtype_code(cdt), n, algo, int(bool(regularise)), nb, m.ptr, m.stride,
                                           o.ptr, o.stride, D.current_stream_ptr(a.device))
        _lib.check(rc, "nfm_batch_inv")
    if copy_back:
        res.copy_(o.tensor)
    return res


def batchmatvec(mat: Tensor, vec: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    """Batched matrix-vector product for small matrices (broadcasting batch dims).

    Reference: _impl/batched.py:154-190.

    Parameters
    ----------
    mat : (..., m, n) tensor
    vec : (..., n) tensor

    Returns
    -------
    matvec : (..., m) tensor
    """
    if (getattr(mat, "requires_grad", False) or getattr(vec, "requires_grad", False)) and torch.is_grad_enabled():
        return A.batchmatvec(mat, vec, out)
    return _batchmatvec(mat, vec, out=out)


def _batchmatvec(mat: Tensor, vec: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    dev = D.common_device(mat, vec)
    if dev.type != "cuda":
        D.check_out_shape(out, (*torch.broadcast_shapes(mat.shape[:-2], vec.shape[:-1]), mat.shape[-2]))
        r = batchmatvec(*_upload(mat, vec))
        if out is not None:
            out.copy_(r)
            return out
        return r.cpu()
    m_, n = mat.shape[-2:]
    if vec.shape[-1] != n:
        raise ValueError(f"mat is (..., {m_}, {n}) but vec is (..., {vec.shape[-1]})")
    cdt = D.compute_dtype(mat, vec)
    batch = tuple(torch.broadcast_shapes(mat.shape[:-2], vec.shape[:-1]))
    nb = D.batch_count(batch)
    o, res, copy_back = D.out_operand(out, (*batch, m_), 1, cdt, dev)
    if nb > 0:
        a = D.as_operand(mat, batch, 2, cdt)
        v = D.as_operand(vec, batch, 1, cdt)
        with D.device_of(dev):
            rc = _lib.load().nfm_batch_matvec(D.dtype_code(cdt), m_, n, nb, a.ptr, a.stride, v.ptr, v.stride,
                                              o.ptr, o.stride, D.current_stream_ptr(dev))
        _lib.check(rc, "nfm_batch_matvec")
    if copy_back:
        res.copy_(o.tensor)
    return res
