"""Drop-in for the LU / Cholesky part of ``nitorch_fastmath.sugar``
(reference: nitorch_fastmath/sugar.py:75-137 lmdiv, :140-191 rmdiv,
:194-258 inv, :261-287 matvec, :290-341 solvevec) for batches of small square
matrices (order <= 10) on CUDA.  Only ``method='lu'`` and ``'chol'`` exist
here: the SVD / pseudo-inverse methods and non-square systems are outside
the hot path (SURVEY.md section 2 row 5) and raise ``NotImplementedError``.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor

from . import _autograd as A
from . import _dispatch as D
from . import _host, _lib
from .batched import batchinv, batchmatvec

__all__ = ['lmdiv', 'rmdiv', 'inv', 'matvec', 'solvevec']


def _algo(method: str) -> int:
    kind = method.lower()
    if kind.startswith('lu'):
        return _lib.ALGO_LU
    if kind.startswith('chol'):
        return _lib.ALGO_LDL
    if kind.startswith(('svd', 'pinv')):
        raise NotImplementedError(f"method {method!r} is outside the B200 hot path (only 'lu' and 'chol')")
    raise ValueError('Unknown inversion method {}.'.format(method))


def lmdiv(a: Tensor, b: Tensor, method: str = 'lu', rcond: float = 1e-15, out: Optional[Tensor] = None) -> Tensor:
    r"""Left matrix division ``inv(a) @ b``  (reference sugar.py:75-137).

    a : `(..., n, n)`, b : `(..., n, k)` -> `(..., n, k)`.  Differentiable in both operands.
    """
    if A.needs_grad(a, b) and torch.is_grad_enabled():
        return A.lmdiv(a, b, method, out)
    return _lmdiv(a, b, method, out)


def _lmdiv(a: Tensor, b: Tensor, method: str = 'lu', out: Optional[Tensor] = None) -> Tensor:
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    if a.shape[-1] != a.shape[-2]:
        raise NotImplementedError("non-square systems (pseudo-inverse) are outside the B200 hot path")
    algo = _algo(method)
    dev = D.common_device(a, b)
    if dev.type != "cuda":
        _host.offload_device()   # raises when there is no CUDA device: no CPU path
        n, k = a.shape[-1], b.shape[-1]
        if b.dim() >= 2 and b.shape[-2] == n:     # anything else is rejected by the device call
            D.check_out_shape(out, (*torch.broadcast_shapes(a.shape[:-2], b.shape[:-2]), n, k))
        plain = (a.dtype == b.dtype and a.dtype in D._DTYPE_CODE and a.is_contiguous() and b.is_contiguous()
                 and 1 <= n <= _lib.MAX_N and b.shape[-2] == n and a.shape[:-2] == b.shape[:-2] and k > 0 and a.numel() > 0
                 and (out is None or (out.device.type == "cpu" and out.is_contiguous() and out.dtype == a.dtype)))
        if plain:
            # dense host batches are streamed through the GPU in chunks (nfm_batch_solve_host)
            code = D.dtype_code(a.dtype)
            nb = a.numel() // (n * n)
            res = out if out is not None else torch.empty(b.shape, dtype=a.dtype, pin_memory=True)
            _host.run_host("nfm_batch_solve_host", code, a.dtype, n * n + n * k, n * k, nb,
                           lambda fn, ws, wsb, chunk, nbuf, streams: fn(code, n, k, algo, nb, a.data_ptr(), b.data_ptr(),
                                                                         res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        return _host.uploaded(lambda da, db: _lmdiv(da, db, method), a, b, out=out)
    n = D.check_order(a.shape[-1])
    if b.shape[-2] != n:
        raise ValueError("a and b have incompatible shapes")
    k = b.shape[-1]
    cdt = D.compute_dtype(a, b)
    batch = tuple(torch.broadcast_shapes(a.shape[:-2], b.shape[:-2]))
    return D.launch("nfm_batch_solve", (n, k, algo), batch, [(a, 2), (b, 2)], rec=(n, k), out=out, dtype=cdt,
                    device=dev, skip_empty=True)


def rmdiv(a: Tensor, b: Tensor, method: str = 'lu', rcond: float = 1e-15, out: Optional[Tensor] = None) -> Tensor:
    r"""Right matrix division ``a @ inv(b)``  (reference sugar.py:140-191, its documented meaning;
    as written the reference returns ``lmdiv(b, a)^T = (inv(b) @ a)^T`` and only runs for square ``a``).

    a : `(..., k, n)`, b : `(..., n, n)` -> `(..., k, n)`.  Solved natively as ``b^T x_r = a_r`` for every
    row ``r`` (``nfm_batch_rsolve``): neither operand is transposed or copied.  Differentiable in both operands.
    """
    if A.needs_grad(a, b) and torch.is_grad_enabled():
        return A.rmdiv(a, b, method, out)
    return _rmdiv(a, b, method, out)


def _rmdiv(a: Tensor, b: Tensor, method: str = 'lu', out: Optional[Tensor] = None) -> Tensor:
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    if b.shape[-1] != b.shape[-2]:
        raise NotImplementedError("non-square systems (pseudo-inverse) are outside the B200 hot path")
    algo = _algo(method)
    dev = D.common_device(a, b)
    if dev.type != "cuda":
        _host.offload_device()   # raises when there is no CUDA device: no CPU path
        if a.dim() >= 2 and a.shape[-1] == b.shape[-1]:     # anything else is rejected by the device call
            D.check_out_shape(out, (*torch.broadcast_shapes(a.shape[:-2], b.shape[:-2]), a.shape[-2], b.shape[-1]))
        return _host.uploaded(lambda da, db: _rmdiv(da, db, method), a, b, out=out)
    n = D.check_order(b.shape[-1])
    if a.shape[-1] != n:
        raise ValueError("a and b have incompatible shapes")
    k = a.shape[-2]
    cdt = D.compute_dtype(a, b)
    batch = tuple(torch.broadcast_shapes(a.shape[:-2], b.shape[:-2]))
    return D.launch("nfm_batch_rsolve", (n, k, algo), batch, [(b, 2), (a, 2)], rec=(k, n), out=out, dtype=cdt,
                    device=dev, skip_empty=True)


def inv(a: Tensor, method: str = 'lu', rcond: float = 1e-15, out: Optional[Tensor] = None) -> Tensor:
    r"""Matrix inversion (reference sugar.py:194-258).  ``'lu'`` is LAPACK
    ``getri`` in the reference, so no closed-form determinant shift here."""
    a = torch.as_tensor(a)
    if a.shape[-1] != a.shape[-2]:
        raise NotImplementedError("non-square systems (pseudo-inverse) are outside the B200 hot path")
    algo = _algo(method)
    return batchinv(a, method='lu' if algo == _lib.ALGO_LU else 'chol', regularise=False, out=out)


def matvec(mat: Tensor, vec: Tensor, out: Optional[Tensor] = None) -> Tensor:
    r"""Matrix-vector product with broadcasting (reference sugar.py:261-287)."""
    return batchmatvec(mat, vec, out=out)


def solvevec(mat: Tensor, vec: Tensor, method: str = 'lu', rcond: float = 1e-15,
             out: Optional[Tensor] = None) -> Tensor:
    r"""Left matrix-vector division ``inv(mat) @ vec``  (reference sugar.py:290-341).

    mat : `(..., n, n)`, vec : `(..., n)` -> `(..., n)`
    """
    vec = torch.as_tensor(vec).unsqueeze(-1)
    if out is not None:
        out = out.unsqueeze(-1)
    return lmdiv(mat, vec, method=method, rcond=rcond, out=out).squeeze(-1)
