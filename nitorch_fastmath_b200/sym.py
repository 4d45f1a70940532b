"""Drop-in for ``nitorch_fastmath.sym`` (reference: nitorch_fastmath/sym.py).

Batches of symmetric matrices stored compactly, coefficient dimension last:
the diagonal first, then the rows of the strict upper triangle::

    [ a d e ]
    [ . b f ]   =>  [a b c d e f]
    [ . . c ]

``sym_matvec`` / ``sym_solve`` also accept (and auto-detect from the trailing
sizes, reference sym.py:16-24) a scaled identity (1 value), a diagonal
(N values) and a full matrix (N*N values).

Every function calls hand-written sm_100a CUDA kernels through the C ABI in
``include/nfm.h``; torch only allocates tensors and supplies the stream.
There is no TorchScript, Triton, cupy or CPU fallback: CUDA tensors run on
their device, CPU tensors are streamed through the current CUDA device, and
without a CUDA device or without the built library every call raises.

Gradients: sym_matvec, sym_addmatvec(_), sym_submatvec(_), sym_solve(_), sym_invert(_)
and sym_det are differentiable (packed, diagonal and scaled-identity layouts), and so
are the Gauss-Newton builders sym_matmul, sym_outer, sym_to_full, sym_matmul_solve and
sym_solve_update(_); the backward passes run on the library's kernels
(``_autograd.py``).  Without a needed gradient each function runs its plain path unchanged.

Signatures are the union of the reference's in-repo implementation
(nitorch_fastmath/_impl/sym.py) and the ``jitfields.sym`` functions that
``nitorch_fastmath.sym`` re-exports (sym.py:30-37).
"""
from __future__ import annotations

import os
from typing import Optional, Sequence, Union

import torch
from torch import Tensor

from . import _autograd as A
from . import _dispatch as D
from . import _host, _lib

__all__ = [
    'sym_to_full', 'sym_diag', 'sym_outer', 'sym_det', 'sym_matmul',
    'sym_matvec',
    'sym_addmatvec', 'sym_addmatvec_',
    'sym_submatvec', 'sym_submatvec_',
    'sym_solve', 'sym_solve_',
    'sym_invert', 'sym_invert_',
    'sym_solve_update', 'sym_solve_update_',     # extensions (not in the reference): fused chains
    'sym_matmul_solve',
]

_METHODS = {None: _lib.ALGO_AUTO, 'auto': _lib.ALGO_AUTO, 'ldl': _lib.ALGO_LDL, 'chol': _lib.ALGO_LDL,
            'lu': _lib.ALGO_LU, 'warp': _lib.ALGO_WARP}


def _algo(method: Optional[str]) -> int:
    if method is None:
        method = os.environ.get("NFM_SYM_METHOD") or None
    try:
        return _METHODS[method.lower() if isinstance(method, str) else method]
    except KeyError:
        raise ValueError(f"unknown method {method!r}; use one of 'auto', 'ldl', 'lu', 'warp'") from None


# ---------------------------------------------------------------------------
# matvec family
# ---------------------------------------------------------------------------

def _matvec(inp: Optional[Tensor], mat: Tensor, vec: Tensor, sign: int,
            dtype: Optional[torch.dtype], out: Optional[Tensor]) -> Tensor:
    if (torch.is_tensor(mat) and torch.is_tensor(vec) and (dtype is None or dtype == vec.dtype)
            and D.plain_cuda(vec, mat, inp, out) and (out is None or out.shape == vec.shape)):
        # fast path: dense CUDA fields with the same batch dims
        n = vec.shape[-1]
        D.check_order(n)
        nn = mat.shape[-1]
        layout = D.detect_layout(nn, n)
        if inp is not None and inp.shape[-1] != n:
            raise ValueError("inp and vec must have the same trailing size")
        res = out if out is not None else D.empty_like_phased(vec)
        nb = vec.numel() // n
        if nb > 0:
            with D.device_of(vec.device):
                rc = _lib.load().nfm_sym_matvec(
                    D.dtype_code(vec.dtype), n, layout, nb, mat.data_ptr(), nn, vec.data_ptr(), n,
                    None if inp is None else inp.data_ptr(), 0 if inp is None else n, sign,
                    res.data_ptr(), n, D.current_stream_ptr(vec.device))
            _lib.check(rc, "nfm_sym_matvec")
        return res
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    tensors = [mat, vec] + ([inp] if inp is not None else [])
    dev = D.common_device(*tensors)
    cdt = D.compute_dtype(*tensors, dtype=dtype)
    n = vec.shape[-1]
    D.check_order(n)
    layout = D.detect_layout(mat.shape[-1], n)
    shapes = [mat.shape[:-1], vec.shape[:-1]] + ([inp.shape[:-1]] if inp is not None else [])
    if inp is not None and inp.shape[-1] != n:
        raise ValueError("inp and vec must have the same trailing size")
    batch = tuple(torch.broadcast_shapes(*shapes))
    nb = D.batch_count(batch)
    code = D.dtype_code(cdt)

    if dev.type != "cuda":
        _host.offload_device()   # raises when there is no CUDA device: no CPU path
        D.check_out_shape(out, (*batch, n))
        plain = (layout == _lib.LAYOUT_SYM and all(_host.is_plain(t) and tuple(t.shape[:-1]) == batch and t.dtype == cdt
                                                   for t in tensors)
                 and (out is None or (_host.is_plain(out) and out.dtype == cdt)))
        if plain and nb > 0:
            res = out if out is not None else torch.empty((*batch, n), dtype=cdt, pin_memory=True)
            nn = mat.shape[-1]
            _host.run_host(
                "nfm_sym_matvec_host", code, cdt, nn + n + (n if inp is not None else 0), n, nb,
                lambda fn, ws, wsb, chunk, nbuf, streams: fn(
                    code, n, nb, mat.data_ptr(), vec.data_ptr(), inp.data_ptr() if inp is not None else None,
                    sign, res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        return _host.uploaded(lambda m, v, i: _matvec(i, m, v, sign, dtype, None), mat, vec, inp, out=out)

    res = D.outer_loop(batch, [(mat, 1), (vec, 1), (inp, 1)], out, (n,), cdt, dev,
                       lambda m, v, i, o: _matvec(i, m, v, sign, cdt, o))
    if res is not None:
        return res
    res = D.launch("nfm_sym_matvec", (n, layout), batch, [(mat, 1), (vec, 1), (inp, 1)], (sign,),
                   rec=(n,), out=out, dtype=cdt, device=dev, struct=True)
    if out is None and dtype is None:
        want = tensors[0].dtype
        for t in tensors[1:]:
            want = torch.promote_types(want, t.dtype)
        if want != res.dtype and want.is_floating_point:   # half / bfloat16 inputs: computed in fp32, returned as promoted
            res = res.to(want)
    return res


def sym_matvec(mat: Tensor, vec: Tensor, dtype: Optional[torch.dtype] = None, out: Optional[Tensor] = None) -> Tensor:
    r"""Matrix-vector product with a compact symmetric matrix: ``mat @ vec``.

    Reference: nitorch_fastmath/_impl/sym.py:134-172 (public name sym.py:30).

    Parameters
    ----------
    mat : `(..., M*(M+1)//2) tensor`
        Compact symmetric matrix (or 1 / M / M*M coefficients: scaled
        identity / diagonal / full).
    vec : `(..., M) tensor`
    dtype, out : optional (jitfields-style)

    Returns
    -------
    matvec : `(..., M) tensor`, dtype = promotion of the inputs
    """
    if A.needs_grad(mat, vec) and torch.is_grad_enabled():
        return A.matvec(None, mat, vec, 0, dtype, out)
    return _matvec(None, mat, vec, 0, dtype, out)


def sym_addmatvec(inp: Tensor, mat: Tensor, vec: Tensor, dtype: Optional[torch.dtype] = None,
                  out: Optional[Tensor] = None) -> Tensor:
    """``inp + mat @ vec``  (reference name: sym.py:31)."""
    if A.needs_grad(inp, mat, vec) and torch.is_grad_enabled():
        return A.matvec(inp, mat, vec, +1, dtype, out)
    return _matvec(torch.as_tensor(inp), mat, vec, +1, dtype, out)


def sym_addmatvec_(inp: Tensor, mat: Tensor, vec: Tensor, dtype: Optional[torch.dtype] = None) -> Tensor:
    """In-place ``inp += mat @ vec``; returns ``inp``  (sym.py:31)."""
    if A.needs_grad(inp, mat, vec) and torch.is_grad_enabled():
        return A.matvec(inp, mat, vec, +1, inp.dtype if dtype is None else dtype, None, inplace=True)
    return _matvec(inp, mat, vec, +1, inp.dtype if dtype is None else dtype, inp)


def sym_submatvec(inp: Tensor, mat: Tensor, vec: Tensor, dtype: Optional[torch.dtype] = None,
                  out: Optional[Tensor] = None) -> Tensor:
    """``inp - mat @ vec``  (sym.py:32)."""
    if A.needs_grad(inp, mat, vec) and torch.is_grad_enabled():
        return A.matvec(inp, mat, vec, -1, dtype, out)
    return _matvec(torch.as_tensor(inp), mat, vec, -1, dtype, out)


def sym_submatvec_(inp: Tensor, mat: Tensor, vec: Tensor, dtype: Optional[torch.dtype] = None) -> Tensor:
    """In-place ``inp -= mat @ vec``; returns ``inp``  (sym.py:32)."""
    if A.needs_grad(inp, mat, vec) and torch.is_grad_enabled():
        return A.matvec(inp, mat, vec, -1, inp.dtype if dtype is None else dtype, None, inplace=True)
    return _matvec(inp, mat, vec, -1, inp.dtype if dtype is None else dtype, inp)


# ---------------------------------------------------------------------------
# solve
# ---------------------------------------------------------------------------

_REG_CACHE = {}   # (values, n, dtype, device) -> device tensor; scalar regularisers recur every iteration


def _as_diag(diag, n: int, dtype: torch.dtype, device: torch.device) -> Optional[Tensor]:
    """Regulariser -> tensor broadcastable to (..., N).  A float or a sequence
    of up to N floats is padded with its last value (reference docstring
    _impl/sym.py:356-357, padding :379-381)."""
    if diag is None:
        return None
    if torch.is_tensor(diag) and diag.dim() >= 1 and diag.shape[-1] in (1, n):
        r = diag.to(device=device, dtype=dtype).expand(*diag.shape[:-1], n)
        # a 1-D regulariser is handed to the library as ONE dense record of n values: a
        # shape-(1,) tensor (stride 0 after expand) or a strided slice must be materialised
        return r if r.dim() > 1 or r.is_contiguous() else r.contiguous()
    key = None
    if isinstance(diag, (int, float)):
        key = ((float(diag),), n, dtype, device)
    elif isinstance(diag, (list, tuple)) and all(isinstance(x, (int, float)) for x in diag):
        key = (tuple(float(x) for x in diag), n, dtype, device)
    if key is not None and key in _REG_CACHE:
        return _REG_CACHE[key]
    e = torch.as_tensor(diag, dtype=dtype).flatten()
    if len(e) > n or len(e) == 0:
        raise ValueError(f"regulariser has {len(e)} entries for a matrix of order {n}")
    e = torch.cat([e, e[-1].expand(n - len(e))]).to(device)
    if key is not None:
        if len(_REG_CACHE) > 256:
            _REG_CACHE.clear()
        _REG_CACHE[key] = e
    return e


def sym_solve(mat: Tensor, vec: Tensor,
              diag: Union[None, float, Sequence[float], Tensor] = None,
              dtype: Optional[torch.dtype] = None, out: Optional[Tensor] = None, *,
              eps: Union[None, float, Sequence[float], Tensor] = None,
              method: Optional[str] = None) -> Tensor:
    r"""Left matrix division for compact symmetric matrices: ``mat \ vec``.

    Reference: nitorch_fastmath/_impl/sym.py:327-398 (public name sym.py:33).
    Orders up to 4 use the reference's closed forms; orders 5..10 factorise
    in registers.  Default (``method='auto'``): LDL^T with a per-matrix pivot
    check and a pivoted-LU fallback, so SPD fields run at LDL^T speed and
    indefinite matrices get the reference's semantics.  ``method='ldl'``:
    unchecked LDL^T; ``'lu'``: partial pivoting for every matrix (what the
    reference does); ``'warp'``: the sub-warp cooperative A/B variant (LDL^T with
    shuffles, no pivoting: SPD input only; several times slower, kept for comparison).

    Parameters
    ----------
    mat : `(..., M*(M+1)//2) tensor`  (or 1 / M / M*M coefficients)
    vec : `(..., M) tensor`
    diag / eps : float, sequence of up to M floats, or `(..., M)` tensor
        Added to the diagonal of ``mat`` (the reference's documented ``eps``;
        as written the reference only runs it for M == 2, see DESIGN.md).
    dtype, out : optional (jitfields-style)

    Returns
    -------
    result : `(..., M) tensor` with ``vec``'s dtype (as the reference).
    """
    if A.needs_grad(mat, vec, diag, eps) and torch.is_grad_enabled():
        return A.solve(mat, vec, diag, dtype, out, eps, method)
    return _solve(mat, vec, diag, dtype, out, eps=eps, method=method)


def _solve(mat: Tensor, vec: Tensor, diag=None, dtype: Optional[torch.dtype] = None, out: Optional[Tensor] = None, *,
           eps=None, method: Optional[str] = None) -> Tensor:
    if eps is not None:
        if diag is not None:
            raise TypeError("give the regulariser as `diag` or as `eps`, not both")
        diag = eps
    if (torch.is_tensor(mat) and torch.is_tensor(vec) and (dtype is None or dtype == vec.dtype)
            and D.plain_cuda(vec, mat, out) and (out is None or out.shape == vec.shape)):
        # fast path: dense CUDA fields with the same batch dims
        n = vec.shape[-1]
        D.check_order(n)
        nn = mat.shape[-1]
        layout = D.detect_layout(nn, n)
        dev = vec.device
        reg = _as_diag(diag, n, vec.dtype, dev)
        if reg is None or reg.dim() == 1 or D.plain_cuda(vec, reg):
            res = out if out is not None else D.empty_like_phased(vec)
            nb = vec.numel() // n
            if nb > 0:
                with D.device_of(dev):
                    rc = _lib.load().nfm_sym_solve(
                        D.dtype_code(vec.dtype), n, layout, _algo(method), nb, mat.data_ptr(), nn, vec.data_ptr(), n,
                        None if reg is None else reg.data_ptr(), 0 if reg is None or reg.dim() == 1 else n,
                        res.data_ptr(), n, D.current_stream_ptr(dev))
                _lib.check(rc, "nfm_sym_solve")
            return res
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    dev = D.common_device(mat, vec)
    cdt = D.compute_dtype(mat, vec, dtype=dtype)
    res_dtype = dtype if dtype is not None else vec.dtype   # reference: result has vec's dtype (half types compute in fp32)
    n = vec.shape[-1]
    D.check_order(n)
    layout = D.detect_layout(mat.shape[-1], n)
    reg = _as_diag(diag, n, cdt, dev)
    shapes = [mat.shape[:-1], vec.shape[:-1]] + ([reg.shape[:-1]] if reg is not None else [])
    batch = tuple(torch.broadcast_shapes(*shapes))
    nb = D.batch_count(batch)
    code = D.dtype_code(cdt)
    algo = _algo(method)

    if dev.type != "cuda":
        _host.offload_device()   # raises when there is no CUDA device: no CPU path
        D.check_out_shape(out, (*batch, n))
        per_voxel_reg = reg is not None and reg.dim() > 1
        plain = (layout == _lib.LAYOUT_SYM and _host.is_plain(mat) and _host.is_plain(vec)
                 and tuple(mat.shape[:-1]) == batch and tuple(vec.shape[:-1]) == batch
                 and mat.dtype == cdt and vec.dtype == cdt and res_dtype == cdt
                 and (reg is None or (per_voxel_reg and _host.is_plain(reg) and tuple(reg.shape[:-1]) == batch))
                 and (out is None or (_host.is_plain(out) and out.dtype == cdt)))
        if plain and nb > 0:
            res = out if out is not None else torch.empty((*batch, n), dtype=cdt, pin_memory=True)
            nn = mat.shape[-1]
            _host.run_host(
                "nfm_sym_solve_host", code, cdt, nn + n + (n if reg is not None else 0), n, nb,
                lambda fn, ws, wsb, chunk, nbuf, streams: fn(
                    code, n, algo, nb, mat.data_ptr(), vec.data_ptr(), reg.data_ptr() if reg is not None else None,
                    res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        return _host.uploaded(lambda m, v, r: _solve(m, v, r, dtype=dtype, method=method), mat, vec, reg, out=out)

    res = D.outer_loop(batch, [(mat, 1), (vec, 1), (reg, 1)], out, (n,), cdt, dev,
                       lambda m, v, r, o: _solve(m, v, r, dtype=cdt, out=o, method=method))
    if res is not None:
        return res if (out is not None or res.dtype == res_dtype) else res.to(res_dtype)
    res = D.launch("nfm_sym_solve", (n, layout, algo), batch, [(mat, 1), (vec, 1), (reg, 1)],
                   rec=(n,), out=out if (out is None or out.dtype == cdt) else None, dtype=cdt, device=dev, struct=True)
    if out is not None and out.dtype != cdt:
        out.copy_(res)
        return out
    if out is None and res.dtype != res_dtype:
        res = res.to(res_dtype)
    return res


def sym_solve_(mat: Tensor, vec: Tensor, diag=None, dtype: Optional[torch.dtype] = None, *,
               eps=None, method: Optional[str] = None) -> Tensor:
    r"""In-place ``vec <- mat \ vec``; returns ``vec``  (reference name sym.py:33)."""
    if A.needs_grad(mat, vec, diag, eps) and torch.is_grad_enabled():
        return A.solve(mat, vec, diag, dtype, None, eps, method, inplace=True)
    return _solve(mat, vec, diag, dtype=dtype, out=vec, eps=eps, method=method)


# ---------------------------------------------------------------------------
# fused solve + update (extension; SURVEY.md section 8f rank 4)
# ---------------------------------------------------------------------------

def sym_solve_update(x: Tensor, mat: Tensor, vec: Tensor, lam: float = 0.0, alpha: float = 1.0,
                     out: Optional[Tensor] = None, *, diag: Optional[Tensor] = None,
                     method: Optional[str] = None) -> Tensor:
    r"""``x - alpha * (mat + lam*I + diag(d)) \ vec`` in one pass over HBM.

    The Gauss-Newton / Levenberg-Marquardt update that otherwise is the chain
    ``step = sym_solve(mat, vec, lam + d); x - alpha * step`` (reference names
    sym.py:31-33); not a function of the reference.  CUDA tensors only;
    ``mat (..., M*(M+1)//2)``, ``vec`` and ``x`` ``(..., M)``; ``diag`` is the
    reference's per-voxel regulariser ``(..., M)`` (or anything broadcastable to it).
    Differentiable with respect to ``x``, ``mat``, ``vec`` and a tensor ``diag``.
    """
    if A.needs_grad(x, mat, vec, diag) and torch.is_grad_enabled():
        return A.solve_update(x, mat, vec, lam, alpha, out, diag, method)
    return _solve_update(x, mat, vec, lam, alpha, out, diag=diag, method=method)


def _solve_update(x: Tensor, mat: Tensor, vec: Tensor, lam: float = 0.0, alpha: float = 1.0,
                  out: Optional[Tensor] = None, *, diag: Optional[Tensor] = None,
                  method: Optional[str] = None) -> Tensor:
    x, mat, vec = torch.as_tensor(x), torch.as_tensor(mat), torch.as_tensor(vec)
    dev = D.common_device(x, mat, vec)
    if dev.type != "cuda":
        raise RuntimeError("sym_solve_update takes CUDA tensors")
    n = vec.shape[-1]
    D.check_order(n)
    if mat.shape[-1] != n * (n + 1) // 2 or x.shape[-1] != n:
        raise ValueError("sym_solve_update takes a packed symmetric mat and x, vec of the same trailing size")
    cdt = D.compute_dtype(x, mat, vec)
    algo = _algo(method)
    if algo not in (_lib.ALGO_AUTO, _lib.ALGO_LDL):
        raise ValueError("sym_solve_update supports method 'auto' or 'ldl'")
    reg = _as_diag(diag, n, cdt, dev)
    shapes = [x.shape[:-1], mat.shape[:-1], vec.shape[:-1]] + ([reg.shape[:-1]] if reg is not None else [])
    batch = tuple(torch.broadcast_shapes(*shapes))
    return D.launch("nfm_sym_solve_update_reg", (n, algo), batch, [(mat, 1), (vec, 1), (x, 1), (reg, 1)],
                    (float(lam), float(alpha)), rec=(n,), out=out, dtype=cdt, device=dev, what="nfm_sym_solve_update")


def sym_solve_update_(x: Tensor, mat: Tensor, vec: Tensor, lam: float = 0.0, alpha: float = 1.0, *,
                      diag: Optional[Tensor] = None, method: Optional[str] = None) -> Tensor:
    r"""In-place ``x -= alpha * (mat + lam*I + diag(d)) \ vec``; returns ``x``."""
    if A.needs_grad(x, mat, vec, diag) and torch.is_grad_enabled():
        return A.solve_update(x, mat, vec, lam, alpha, None, diag, method, inplace=True)
    return _solve_update(x, mat, vec, lam, alpha, out=x, diag=diag, method=method)


def _mode(k: int, d: int) -> int:
    """C ABI ``mode`` of the J/H products: 1 (J H J^T) for k == d <= 3, the reference's unrolled
    branches (_impl/sym.py:532-593); 0 (J^T H J) otherwise."""
    return 1 if (k == d and k <= 3) else 0


def _packed_h(j: Tensor, h: Tensor) -> Tensor:
    """A diagonal Hessian (k values; reference jhjn accepts it: _impl/sym.py:603-606) in packed form with
    zero off-diagonals.  The autograd wrappers pad it before their Function, so that its gradient is
    the diagonal of the packed one (the backward of torch.cat)."""
    k = j.shape[-2]
    if h.shape[-1] == k and k > 1:
        return torch.cat([h, h.new_zeros((*h.shape[:-1], k * (k - 1) // 2))], -1)
    return h


def sym_matmul_solve(j: Tensor, h: Tensor, g: Tensor, diag=None, out: Optional[Tensor] = None) -> Tensor:
    r"""``(J^T H J + diag(d)) \ g`` with the packed Hessian built and solved in registers.

    The fused form of the Gauss-Newton chain ``sym_solve(sym_matmul(j, h), g, diag)``
    (reference _impl/sym.py:637-670 then :327-398): the ``d*(d+1)//2``-coefficient Hessian
    field is never written to memory.  ``j (..., k, d)``, ``h (..., k*(k+1)//2)`` or
    diagonal ``(..., k)``, ``g (..., d)``, ``diag`` float / sequence / ``(..., d)``;
    ``1 <= k, d <= 6`` or ``k <= 10`` with ``d <= 3``; CUDA tensors.  Like ``sym_matmul`` it evaluates ``J H J^T``
    for ``k == d <= 3`` (the reference's unrolled branches).  Not a function of the reference.
    Differentiable with respect to ``j``, ``h``, ``g`` and a tensor ``diag``.
    """
    if A.needs_grad(j, h, g, diag) and torch.is_grad_enabled():
        return A.matmul_solve(j, h, g, diag, out)
    return _matmul_solve(j, h, g, diag, out)


def _matmul_solve(j: Tensor, h: Tensor, g: Tensor, diag=None, out: Optional[Tensor] = None) -> Tensor:
    j, h, g = torch.as_tensor(j), torch.as_tensor(h), torch.as_tensor(g)
    dev = D.common_device(j, h, g)
    if dev.type != "cuda":
        raise RuntimeError("sym_matmul_solve takes CUDA tensors")
    k, d = j.shape[-2:]
    if not ((1 <= k <= 6 and 1 <= d <= 6) or (1 <= k <= _lib.MAX_N and 1 <= d <= 3)):
        raise ValueError("sym_matmul_solve supports 1 <= k, d <= 6, or k <= 10 with d <= 3 (use sym_matmul + sym_solve otherwise)")
    h = _packed_h(j, h)
    if h.shape[-1] != k * (k + 1) // 2:
        raise ValueError("h must be compact symmetric (k*(k+1)//2 coefficients) or diagonal (k coefficients)")
    if g.shape[-1] != d:
        raise ValueError(f"g must have {d} trailing values")
    cdt = D.compute_dtype(j, h, g)
    reg = _as_diag(diag, d, cdt, dev)
    shapes = [j.shape[:-2], h.shape[:-1], g.shape[:-1]] + ([reg.shape[:-1]] if reg is not None else [])
    batch = tuple(torch.broadcast_shapes(*shapes))
    return D.launch("nfm_sym_matmul_solve", (k, d, _mode(k, d)), batch, [(j, 2), (h, 1), (g, 1), (reg, 1)],
                    rec=(d,), out=out, dtype=cdt, device=dev)


# ---------------------------------------------------------------------------
# invert
# ---------------------------------------------------------------------------

def sym_invert(mat: Tensor, diag: bool = False, dtype: Optional[torch.dtype] = None,
               out: Optional[Tensor] = None, *, method: Optional[str] = None) -> Tensor:
    r"""Matrix inversion for compact symmetric matrices.

    Reference: nitorch_fastmath/_impl/sym.py:455-493 (public name sym.py:34).

    Parameters
    ----------
    mat : `(..., M*(M+1)//2) tensor`
    diag : bool, default=False
        If True, only return the diagonal of the inverse.

    Returns
    -------
    imat : `(..., M or M*(M+1)//2) tensor` (compact storage, same ordering)
    """
    if A.needs_grad(mat) and torch.is_grad_enabled():
        return A.invert(mat, diag, dtype, out, method)
    return _invert(mat, diag, dtype, out, method=method)


def _invert(mat: Tensor, diag: bool = False, dtype: Optional[torch.dtype] = None,
            out: Optional[Tensor] = None, *, method: Optional[str] = None) -> Tensor:
    if _algo(method) == _lib.ALGO_WARP:
        raise ValueError("method='warp' is a sym_solve A/B kernel (SPD input, no pivoting); sym_invert has no such variant")
    if dtype is None and torch.is_tensor(mat) and D.plain_cuda(mat) and (
            out is None or (D.plain_cuda(mat, out) and out.shape[-1] == (D.packed_order(mat.shape[-1]) if diag else mat.shape[-1]))):
        nn = mat.shape[-1]
        n = D.packed_order(nn)
        D.check_order(n)
        no = n if diag else nn
        res = out if out is not None else (D.empty_like_phased(mat) if no == nn else
                                           torch.empty((*mat.shape[:-1], no), dtype=mat.dtype, device=mat.device))
        nb = mat.numel() // nn
        if nb > 0:
            with D.device_of(mat.device):
                rc = _lib.load().nfm_sym_invert(D.dtype_code(mat.dtype), n, _algo(method), int(bool(diag)), nb,
                                                mat.data_ptr(), nn, res.data_ptr(), no, D.current_stream_ptr(mat.device))
            _lib.check(rc, "nfm_sym_invert")
        return res
    mat = torch.as_tensor(mat)
    dev = mat.device
    cdt = D.compute_dtype(mat, dtype=dtype)
    nn = mat.shape[-1]
    n = D.packed_order(nn)
    D.check_order(n)
    no = n if diag else nn
    batch = tuple(mat.shape[:-1])
    nb = D.batch_count(batch)
    code = D.dtype_code(cdt)
    algo = _algo(method)

    if dev.type != "cuda":
        _host.offload_device()   # raises when there is no CUDA device: no CPU path
        D.check_out_shape(out, (*batch, no))
        plain = (_host.is_plain(mat) and mat.dtype == cdt
                 and (out is None or (_host.is_plain(out) and out.dtype == cdt)))
        if plain and nb > 0:
            res = out if out is not None else torch.empty((*batch, no), dtype=cdt, pin_memory=True)
            _host.run_host(
                "nfm_sym_invert_host", code, cdt, nn, no, nb,
                lambda fn, ws, wsb, chunk, nbuf, streams: fn(
                    code, n, algo, int(bool(diag)), nb, mat.data_ptr(), res.data_ptr(), ws, wsb, chunk, nbuf, streams))
            return res
        return _host.uploaded(lambda m: _invert(m, diag, dtype=dtype, method=method), mat, out=out)

    res = D.launch("nfm_sym_invert", (n, algo, int(bool(diag))), batch, [(mat, 1)], rec=(no,), out=out,
                   dtype=cdt, device=dev, struct=True)
    if out is None and dtype is None and mat.dtype != res.dtype and mat.dtype.is_floating_point:
        res = res.to(mat.dtype)
    return res


def sym_invert_(mat: Tensor, dtype: Optional[torch.dtype] = None, *, method: Optional[str] = None) -> Tensor:
    """In-place inversion; returns ``mat``  (reference name sym.py:34)."""
    if A.needs_grad(mat) and torch.is_grad_enabled():
        return A.invert(mat, False, dtype, None, method, inplace=True)
    return _invert(mat, False, dtype=dtype, out=mat, method=method)


# ---------------------------------------------------------------------------
# remaining public names of nitorch_fastmath/sym.py:29
# ---------------------------------------------------------------------------

def sym_to_full(mat: Tensor) -> Tensor:
    """Compact symmetric -> full `(..., M, M)`  (reference _impl/sym.py:16-60)."""
    if A.needs_grad(mat) and torch.is_grad_enabled():
        return A.to_full(mat)
    return _to_full(mat)


def _to_full(mat: Tensor) -> Tensor:
    mat = torch.as_tensor(mat)
    n = D.check_order(D.packed_order(mat.shape[-1]))
    if mat.device.type != "cuda":
        return _host.uploaded(_to_full, mat)
    return D.launch("nfm_sym_to_full", (n,), tuple(mat.shape[:-1]), [(mat, 1)], rec=(n, n),
                    dtype=D.compute_dtype(mat), device=mat.device)


def sym_diag(mat: Tensor) -> Tensor:
    """View into the main diagonal `(..., M)`  (reference _impl/sym.py:63-84)."""
    mat = torch.as_tensor(mat)
    return mat[..., :D.packed_order(mat.shape[-1])]


def sym_outer(x: Tensor) -> Tensor:
    """Symmetric outer product ``x x^T`` in compact storage (reference _impl/sym.py:496-528)."""
    if A.needs_grad(x) and torch.is_grad_enabled():
        return A.outer(x)
    return _outer(x)


def _outer(x: Tensor) -> Tensor:
    x = torch.as_tensor(x)
    n = D.check_order(x.shape[-1])
    if x.device.type != "cuda":
        return _host.uploaded(_outer, x)
    return D.launch("nfm_sym_outer", (n,), tuple(x.shape[:-1]), [(x, 1)], rec=(n * (n + 1) // 2,),
                    dtype=D.compute_dtype(x), device=x.device)


def sym_det(mat: Tensor) -> Tensor:
    """Determinant of a compact symmetric matrix `(...)`  (reference _impl/sym.py:401-452;
    the reference's batched N >= 3 result is wrong (:434), this one is not)."""
    if A.needs_grad(mat) and torch.is_grad_enabled():
        return A.det(mat)
    return _det(mat)


def _det(mat: Tensor) -> Tensor:
    mat = torch.as_tensor(mat)
    n = D.check_order(D.packed_order(mat.shape[-1]))
    if mat.device.type != "cuda":
        return _host.uploaded(_det, mat)
    return D.launch("nfm_sym_det", (n,), tuple(mat.shape[:-1]), [(mat, 1)], rec=(),
                    dtype=D.compute_dtype(mat), device=mat.device)


def sym_matmul(j: Tensor, h: Tensor) -> Tensor:
    r"""Symmetric product :math:`J^T H J` with compact ``h`` and compact result.

    Reference: nitorch_fastmath/_impl/sym.py:637-670.  ``j`` is `(..., k, d)`,
    ``h`` `(..., k*(k+1)//2)`, result `(..., d*(d+1)//2)`.  Note that for
    ``k == d <= 3`` the reference's unrolled branches (:532-593) evaluate
    :math:`J H J^T`; this drop-in reproduces that (C ABI ``mode=1``).
    Differentiable with respect to ``j`` and ``h`` (also a diagonal ``h``).
    """
    if A.needs_grad(j, h) and torch.is_grad_enabled():
        return A.matmul(j, h)
    return _matmul(j, h)


def _matmul(j: Tensor, h: Tensor) -> Tensor:
    j, h = torch.as_tensor(j), torch.as_tensor(h)
    dev = D.common_device(j, h)
    if dev.type != "cuda":
        return _host.uploaded(_matmul, j, h)
    k, d = j.shape[-2:]
    if not (1 <= k <= _lib.MAX_N and 1 <= d <= _lib.MAX_N):
        raise ValueError(f"sym_matmul supports 1 <= k, d <= {_lib.MAX_N}")
    h = _packed_h(j, h)
    if h.shape[-1] != k * (k + 1) // 2:
        raise ValueError("h must be compact symmetric (k*(k+1)//2 coefficients) or diagonal (k coefficients)")
    cdt = h.dtype if h.dtype in (torch.float32, torch.float64) else D.compute_dtype(j, h)
    batch = tuple(torch.broadcast_shapes(j.shape[:-2], h.shape[:-1]))
    return D.launch("nfm_sym_matmul", (k, d, _mode(k, d)), batch, [(j, 2), (h, 1)], rec=(d * (d + 1) // 2,),
                    dtype=cdt, device=dev)
