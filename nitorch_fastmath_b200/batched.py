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
    return D.check_order(a.shape[-1])


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
    if A.needs_grad(a) and torch.is_grad_enabled():
        return A.batchdet(a, out)
    return _batchdet(a, out=out)


def _batchdet(a: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    a = torch.as_tensor(a)
    n = _square_order(a)
    if a.device.type != "cuda":
        nb = a.numel() // (n * n)
        D.check_out_shape(out, a.shape[:-2])
        if _plain_host(a) and nb > 0 and (out is None or _plain_host(a, out)):
            code = D.dtype_code(a.dtype)
            res = out if out is not None else torch.empty(a.shape[:-2], dtype=a.dtype, pin_memory=True)
            _host.run_host("nfm_batch_det_host", code, a.dtype, n * n, 1, nb,
                           lambda fn, ws, wsb, chunk, nbuf, streams: fn(code, n, nb, a.data_ptr(), res.data_ptr(), ws, wsb,
                                                                         chunk, nbuf, streams))
            return res
        return _host.uploaded(_batchdet, a, out=out)
    return D.launch("nfm_batch_det", (n,), tuple(a.shape[:-2]), [(a, 2)], rec=(), out=out,
                    dtype=D.compute_dtype(a), device=a.device)


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
    if A.needs_grad(a) and torch.is_grad_enabled():
        return A.batchinv(a, method, regularise, out)
    return _batchinv(a, method=method, regularise=regularise, out=out)


def _batchinv(a: Tensor, *, method: str = 'auto', regularise: bool = True, out: Optional[Tensor] = None) -> Tensor:
    a = torch.as_tensor(a)
    kind = method.lower()
    algo = {'auto': _lib.ALGO_AUTO, 'lu': _lib.ALGO_LU, 'chol': _lib.ALGO_LDL, 'ldl': _lib.ALGO_LDL}.get(kind)
    if algo is None:
        raise ValueError(f"unknown method {method!r}")
    n = _square_order(a)
    if a.device.type != "cuda":
        nb = a.numel() // (n * n)
        D.check_out_shape(out, a.shape)
        if _plain_host(a) and nb > 0 and (out is None or _plain_host(a, out)):
            code = D.dtype_code(a.dtype)
            res = out if out is not None else torch.empty(a.shape, dtype=a.dtype, pin_memory=True)
            _host.run_host("nfm_batch_inv_host", code, a.dtype, n * n, n * n, nb,
                           lambda fn, ws, wsb, chunk, nbuf, streams: fn(code, n, algo, int(bool(regularise)), nb, a.data_ptr(),
                                                                         res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        return _host.uploaded(lambda m: _batchinv(m, method=method, regularise=regularise), a, out=out)
    return D.launch("nfm_batch_inv", (n, algo, int(bool(regularise))), tuple(a.shape[:-2]), [(a, 2)], rec=(n, n),
                    out=out, dtype=D.compute_dtype(a), device=a.device)


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
    if A.needs_grad(mat, vec) and torch.is_grad_enabled():
        return A.batchmatvec(mat, vec, out)
    return _batchmatvec(mat, vec, out=out)


def _batchmatvec(mat: Tensor, vec: Tensor, *, out: Optional[Tensor] = None) -> Tensor:
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    dev = D.common_device(mat, vec)
    if dev.type != "cuda":
        D.check_out_shape(out, (*torch.broadcast_shapes(mat.shape[:-2], vec.shape[:-1]), mat.shape[-2]))
        return _host.uploaded(_batchmatvec, mat, vec, out=out)
    m_, n = mat.shape[-2:]
    if vec.shape[-1] != n:
        raise ValueError(f"mat is (..., {m_}, {n}) but vec is (..., {vec.shape[-1]})")
    cdt = D.compute_dtype(mat, vec)
    batch = tuple(torch.broadcast_shapes(mat.shape[:-2], vec.shape[:-1]))
    return D.launch("nfm_batch_matvec", (m_, n), batch, [(mat, 2), (vec, 1)], rec=(m_,), out=out, dtype=cdt, device=dev)
