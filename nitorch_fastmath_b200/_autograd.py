"""Gradients of the packed-symmetric routines (sym_matvec family, sym_solve,
sym_invert, sym_det), of the Gauss-Newton builders (sym_matmul, sym_outer,
sym_to_full, sym_matmul_solve, sym_solve_update(_)) and of the dense ones
(batchdet, batchinv, batchmatvec, lmdiv, rmdiv; through them inv, solvevec and matvec).

The public functions in ``sym.py``, ``batched.py`` and ``sugar.py`` route here
only when grad mode is on and a tensor operand requires grad; otherwise they run
their plain path untouched.
Each ``torch.autograd.Function`` runs the plain implementation in ``forward``
and the library's backward kernels (``nfm_sym_outer2``,
``nfm_sym_invert_backward``, ``nfm_sym_det_backward``, plus the forward
``nfm_sym_matvec`` / ``nfm_sym_solve`` for the vector gradients) in
``backward``, on the current stream.  torch allocates, casts between the
compute dtype and the operands' dtypes, and sums a gradient over the batch
dimensions its operand was broadcast along (``sum_to_size``).

Notation (DESIGN.md, "Gradients"): p = the stored coefficients of A, g = the
incoming gradient, S(u, w) = the gradient of u^T A w with respect to p.

  y = inp +/- A v        d_inp = g, d_v = +/- A g, d_p = +/- S(g, v)
  x = (A + diag d)^-1 v  u = (A + diag d)^-1 g: d_v = u, d_p = -S(u, x), d_d = -u * x
  B = A^-1               d_p from M = B G B (nfm_sym_invert_backward)
  t = det A              d_p = g * adjugate, off-diagonal doubled (nfm_sym_det_backward)

Gauss-Newton builders (G^ = the full symmetric form of a packed gradient with the
off-diagonals halved, pack(M) = M_ii, 2 M_ij):

  Y = J^T H J            dJ = 2 H J G^, dH = pack(J G^ J^T)     (nfm_sym_matmul_backward)
  Y = J H J^T (k=d<=3)   dJ = 2 G^ J H, dH = pack(J^T G^ J)
  y = x x^T              dx = 2 G^ x                            (nfm_sym_outer_backward)
  F = sym_to_full(p)     dp_ii = G_ii, dp_ij = G_ij + G_ji      (nfm_sym_to_full_backward)
  x = (J^T H J + diag d)^-1 g0, out = x - alpha (A + lam I + diag d)^-1 v: chains of
                         nfm_sym_matmul, nfm_sym_solve, nfm_sym_outer2 and the matmul backward

Dense (G = the incoming gradient; for method 'chol' the symmetric part of each matrix
gradient, torch's convention for cholesky + cholesky_solve / cholesky_inverse):

  t = det A              dA = g adj(A)^T                       (nfm_batch_det_backward)
  Y = A^-1               dA = -Y^T G Y^T                       (nfm_batch_inv_backward)
  X = A^-1 B             U = A^-T G: dB = U, dA = -U X^T       (nfm_batch_tsolve, nfm_batch_outer)
  Y = B A^-1             U = G A^-T: dB = U, dA = -Y^T U
  y = A v                dA = g v^T, dv = A^T g                (nfm_batch_outer, nfm_batch_tmatvec)

Backward passes are once-differentiable: a second-order gradient raises.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import torch
from torch import Tensor
from torch.autograd.function import once_differentiable

from . import _dispatch as D
from . import _host, _lib
from . import batched as B
from . import sym as S


def needs_grad(*operands) -> bool:
    for t in operands:
        if getattr(t, "requires_grad", False):
            return True
    return False


def _layout_len(layout: int, n: int) -> int:
    return {_lib.LAYOUT_SCALED_IDENTITY: 1, _lib.LAYOUT_DIAG: n, _lib.LAYOUT_SYM: n * (n + 1) // 2}[layout]


def outer2(u: Tensor, w: Tensor, layout: int, sign: int) -> Tensor:
    """``sign * S(u, w)`` in ``layout``: records of 1 / N / N(N+1)/2 over the broadcast batch of u, w."""
    n = u.shape[-1]
    batch = tuple(torch.broadcast_shapes(u.shape[:-1], w.shape[:-1]))
    return D.launch("nfm_sym_outer2", (n, layout), batch, [(u, 1), (w, 1)], (sign,), rec=(_layout_len(layout, n),),
                    dtype=u.dtype, device=u.device, skip_empty=True)


def invert_backward(inv: Tensor, grad: Tensor, diag_only: bool) -> Tensor:
    """Gradient of ``sym_invert`` with respect to the packed matrix, from the packed inverse."""
    nn = inv.shape[-1]
    n = D.packed_order(nn)
    batch = tuple(torch.broadcast_shapes(inv.shape[:-1], grad.shape[:-1]))
    return D.launch("nfm_sym_invert_backward", (n, int(bool(diag_only))), batch, [(inv, 1), (grad, 1)], rec=(nn,),
                    dtype=inv.dtype, device=inv.device, skip_empty=True)


def det_backward(mat: Tensor, grad: Tensor) -> Tensor:
    """Gradient of ``sym_det`` with respect to the packed matrix; ``grad`` has the batch shape."""
    nn = mat.shape[-1]
    batch = tuple(torch.broadcast_shapes(mat.shape[:-1], grad.shape))
    return D.launch("nfm_sym_det_backward", (D.packed_order(nn),), batch, [(mat, 1), (grad.unsqueeze(-1), 1)], rec=(nn,),
                    dtype=mat.dtype, device=mat.device, skip_empty=True)


def _work_device(dev: torch.device) -> torch.device:
    """CPU operands compute their gradients on the CUDA device their forward streamed through."""
    return dev if dev.type == "cuda" else _host.offload_device()


def _grad_for(grad: Optional[Tensor], like: Tensor) -> Optional[Tensor]:
    """Sum over the dims ``like`` was broadcast along, back to its dtype and device."""
    if grad is None:
        return None
    if tuple(grad.shape) != tuple(like.shape):
        grad = grad.sum_to_size(like.shape)
    return grad.to(device=like.device, dtype=like.dtype)


def _check_layout(layout: int, what: str, *operands) -> None:
    """A full N*N `mat` is a general matrix to the kernels: its gradients (and those of the vector and the
    regulariser of a solve) would need transposed products and solves."""
    if layout == _lib.LAYOUT_FULL and needs_grad(*operands):
        raise NotImplementedError(f"{what}: gradients with a full (N*N) matrix are not supported; "
                                  "use the packed, diagonal or scaled-identity layout")


def _check_out(out: Optional[Tensor], what: str) -> None:
    if out is not None:
        raise RuntimeError(f"{what}(): functions with out=... arguments don't support automatic differentiation, "
                           "but one of the arguments requires grad")


# ---------------------------------------------------------------------------
# matvec family:  y = [inp +/-] A v
# ---------------------------------------------------------------------------

class _Matvec(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inp, mat, vec, sign, dtype, inplace):
        res = S._matvec(inp, mat, vec, sign, dtype, inp if inplace else None)
        if inplace:
            ctx.mark_dirty(inp)
        ctx.save_for_backward(mat, vec)
        ctx.sign = sign
        ctx.cdt = D.compute_dtype(*[t for t in (mat, vec, inp) if t is not None], dtype=dtype)
        ctx.inp_meta = None if inp is None else (inp.shape, inp.dtype, inp.device)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        mat, vec = ctx.saved_tensors
        need_inp, need_mat, need_vec = ctx.needs_input_grad[:3]
        dev = _work_device(vec.device)
        cdt = ctx.cdt
        n = vec.shape[-1]
        g = g.to(device=dev, dtype=cdt)
        d_inp = d_mat = d_vec = None
        if need_inp:
            shape, dt, idev = ctx.inp_meta
            d_inp = g.sum_to_size(shape) if tuple(g.shape) != tuple(shape) else g
            d_inp = d_inp.to(device=idev, dtype=dt)
        if need_vec:
            m = mat.to(device=dev, dtype=cdt)
            if ctx.sign < 0:   # -A g as 0 - A g: a broadcast zero addend, no extra pass
                d_vec = S._matvec(torch.zeros(n, dtype=cdt, device=dev), m, g, -1, cdt, None)
            else:
                d_vec = S._matvec(None, m, g, 0, cdt, None)
            d_vec = _grad_for(d_vec, vec)
        if need_mat:
            layout = D.detect_layout(mat.shape[-1], n)
            d_mat = _grad_for(outer2(g, vec.to(device=dev, dtype=cdt), layout, -1 if ctx.sign < 0 else 1), mat)
        return d_inp, d_mat, d_vec, None, None, None


def matvec(inp, mat, vec, sign: int, dtype, out, inplace: bool = False) -> Tensor:
    what = {0: "sym_matvec", 1: "sym_addmatvec", -1: "sym_submatvec"}[sign] + ("_" if inplace else "")
    _check_out(out, what)
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    inp = None if inp is None else torch.as_tensor(inp)
    _check_layout(D.detect_layout(mat.shape[-1], vec.shape[-1]), what, mat, vec)
    return _Matvec.apply(inp, mat, vec, sign, dtype, inplace)


# ---------------------------------------------------------------------------
# solve:  x = (A + diag d)^-1 v
# ---------------------------------------------------------------------------

class _Solve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mat, vec, diag, dtype, method, inplace):
        res = S._solve(mat, vec, diag, dtype=dtype, out=vec if inplace else None, method=method)
        if inplace:
            ctx.mark_dirty(vec)
        reg_t = diag if torch.is_tensor(diag) else None
        ctx.save_for_backward(mat, res, reg_t)
        ctx.reg = None if reg_t is not None else diag   # scalar / sequence regulariser: no gradient
        ctx.method = method
        ctx.cdt = D.compute_dtype(mat, vec, dtype=dtype)
        ctx.vec_meta = (vec.shape, vec.dtype, vec.device)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        mat, x, reg_t = ctx.saved_tensors
        need_mat, need_vec, need_diag = ctx.needs_input_grad[:3]
        dev = _work_device(mat.device)
        cdt = ctx.cdt
        m = mat.to(device=dev, dtype=cdt)
        reg = reg_t.to(device=dev) if reg_t is not None else ctx.reg
        u = S._solve(m, g.to(device=dev, dtype=cdt), reg, dtype=cdt, method=ctx.method)
        d_mat = d_vec = d_diag = None
        if need_vec:
            shape, dt, vdev = ctx.vec_meta
            d_vec = (u.sum_to_size(shape) if tuple(u.shape) != tuple(shape) else u).to(device=vdev, dtype=dt)
        if need_mat or need_diag:
            xc = x.to(device=dev, dtype=cdt)
            layout = D.detect_layout(mat.shape[-1], x.shape[-1])
            full = outer2(u, xc, layout, -1) if need_mat else None
            if need_mat:
                d_mat = _grad_for(full, mat)
            if need_diag:
                # -u * x, the diagonal part of d_p: the D-layout record is that already
                dd = full if layout == _lib.LAYOUT_DIAG and full is not None else outer2(u, xc, _lib.LAYOUT_DIAG, -1)
                d_diag = _grad_for(dd, reg_t)
        return d_mat, d_vec, d_diag, None, None, None


def solve(mat, vec, diag, dtype, out, eps, method, inplace: bool = False) -> Tensor:
    what = "sym_solve_" if inplace else "sym_solve"
    _check_out(out, what)
    if eps is not None:
        if diag is not None:
            raise TypeError("give the regulariser as `diag` or as `eps`, not both")
        diag = eps
    mat, vec = torch.as_tensor(mat), torch.as_tensor(vec)
    _check_layout(D.detect_layout(mat.shape[-1], vec.shape[-1]), what, mat, vec, diag)
    return _Solve.apply(mat, vec, diag, dtype, method, inplace)


# ---------------------------------------------------------------------------
# invert:  B = A^-1  (or diag(A^-1))
# ---------------------------------------------------------------------------

class _Invert(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mat, diag, dtype, method, inplace):
        res = S._invert(mat, diag, dtype, mat if inplace else None, method=method)
        if inplace:
            ctx.mark_dirty(mat)
        # the diagonal-only forward does not produce the packed inverse the backward needs:
        # keep A and invert it again in backward
        ctx.save_for_backward(mat if diag else res)
        ctx.diag = bool(diag)
        ctx.method = method
        ctx.cdt = D.compute_dtype(mat, dtype=dtype)
        ctx.mat_meta = (mat.shape, mat.dtype, mat.device)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        saved, = ctx.saved_tensors
        _, dt, mdev = ctx.mat_meta
        dev = _work_device(mdev)
        cdt = ctx.cdt
        inv = saved.to(device=dev, dtype=cdt)
        if ctx.diag:
            inv = S._invert(inv, False, cdt, method=ctx.method)
        d = invert_backward(inv, g.to(device=dev, dtype=cdt), ctx.diag)
        return d.to(device=mdev, dtype=dt), None, None, None, None


def invert(mat, diag, dtype, out, method, inplace: bool = False) -> Tensor:
    _check_out(out, "sym_invert_" if inplace else "sym_invert")
    return _Invert.apply(torch.as_tensor(mat), diag, dtype, method, inplace)


# ---------------------------------------------------------------------------
# det:  t = det A
# ---------------------------------------------------------------------------

class _Det(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mat):
        ctx.save_for_backward(mat)
        return S._det(mat)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        mat, = ctx.saved_tensors
        dev = _work_device(mat.device)
        cdt = D.compute_dtype(mat)
        d = det_backward(mat.to(device=dev, dtype=cdt), g.to(device=dev, dtype=cdt))
        return d.to(device=mat.device, dtype=mat.dtype)


def det(mat) -> Tensor:
    return _Det.apply(torch.as_tensor(mat))


# ---------------------------------------------------------------------------
# dense routines: records (..., n, n), (..., n, k), (..., k, n), (..., n)
# ---------------------------------------------------------------------------

def _meta(t: Tensor) -> SimpleNamespace:
    """What ``_grad_for`` needs of an operand, without keeping it alive."""
    return SimpleNamespace(shape=t.shape, dtype=t.dtype, device=t.device)


def _batch(*records) -> tuple:
    return tuple(torch.broadcast_shapes(*[t.shape[:t.dim() - nd] for t, nd in records]))


def dense_det_backward(a: Tensor, g: Tensor) -> Tensor:
    """g * adj(A)^T for (..., n, n) matrices and (...) incoming gradients."""
    n = a.shape[-1]
    batch = _batch((a, 2), (g, 0))
    return D.launch("nfm_batch_det_backward", (n,), batch, [(a.flatten(-2), 1), (g.unsqueeze(-1), 1)], rec=(n * n,),
                    dtype=a.dtype, device=a.device, skip_empty=True).view(*batch, n, n)


def dense_inv_backward(y: Tensor, g: Tensor, sym: bool) -> Tensor:
    """-Y^T G Y^T, or -Y (G + G^T) Y / 2 when ``sym``, from the inverse Y."""
    n = y.shape[-1]
    batch = _batch((y, 2), (g, 2))
    return D.launch("nfm_batch_inv_backward", (n, int(sym)), batch, [(y.flatten(-2), 1), (g.flatten(-2), 1)],
                    rec=(n * n,), dtype=y.dtype, device=y.device, skip_empty=True).view(*batch, n, n)


def dense_outer(u: Tensor, w: Tensor, rows: bool, sym: bool, sign: int) -> Tensor:
    """``sign * U W^T`` (U: (..., m, k), W: (..., n, k)) or, with ``rows``, ``sign * U^T W``
    (U: (..., k, m), W: (..., k, n)); the symmetric part when ``sym``."""
    k, m = (u.shape[-2], u.shape[-1]) if rows else (u.shape[-1], u.shape[-2])
    n = w.shape[-1] if rows else w.shape[-2]
    batch = _batch((u, 2), (w, 2))
    if k == 0:
        return torch.zeros((*batch, m, n), dtype=u.dtype, device=u.device)
    return D.launch("nfm_batch_outer", (m, n, k, int(rows), int(sym), sign), batch,
                    [(u.flatten(-2), 1), (w.flatten(-2), 1)], rec=(m * n,), dtype=u.dtype, device=u.device,
                    skip_empty=True).view(*batch, m, n)


def dense_tsolve(a: Tensor, b: Tensor, right: bool, algo: int) -> Tensor:
    """``A^-T B`` (B: (..., n, k)) or, with ``right``, ``B A^-T`` (B: (..., k, n))."""
    n = a.shape[-1]
    k = b.shape[-2] if right else b.shape[-1]
    batch = _batch((a, 2), (b, 2))
    return D.launch("nfm_batch_tsolve", (n, k, int(right), algo), batch, [(a.flatten(-2), 1), (b.flatten(-2), 1)],
                    rec=(n * k,), dtype=a.dtype, device=a.device, skip_empty=True).view(*batch, *b.shape[-2:])


def dense_tmatvec(a: Tensor, v: Tensor) -> Tensor:
    """``A^T v`` for A: (..., m, n), v: (..., m)."""
    m, n = a.shape[-2:]
    batch = _batch((a, 2), (v, 1))
    return D.launch("nfm_batch_tmatvec", (m, n), batch, [(a.flatten(-2), 1), (v, 1)], rec=(n,), dtype=a.dtype,
                    device=a.device, skip_empty=True)


class _BatchDet(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a):
        ctx.save_for_backward(a)
        return B._batchdet(a)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, = ctx.saved_tensors
        dev, cdt = _work_device(a.device), D.compute_dtype(a)
        return _grad_for(dense_det_backward(a.to(device=dev, dtype=cdt), g.to(device=dev, dtype=cdt)), a)


def batchdet(a, out) -> Tensor:
    _check_out(out, "batchdet")
    return _BatchDet.apply(torch.as_tensor(a))


class _BatchInv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, method, regularise):
        res = B._batchinv(a, method=method, regularise=regularise)
        # n = 2, 3 with `regularise`: the determinant shift is a constant, the gradient is that of the returned Y
        ctx.save_for_backward(res)
        ctx.sym = method.lower() in ("chol", "ldl")
        ctx.a = _meta(a)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        y, = ctx.saved_tensors
        dev = _work_device(y.device)
        d = dense_inv_backward(y.to(device=dev), g.to(device=dev, dtype=y.dtype), ctx.sym)
        return _grad_for(d, ctx.a), None, None


def batchinv(a, method, regularise, out) -> Tensor:
    _check_out(out, "batchinv")
    return _BatchInv.apply(torch.as_tensor(a), method, regularise)


class _BatchMatvec(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mat, vec):
        ctx.save_for_backward(mat, vec)
        return B._batchmatvec(mat, vec)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        mat, vec = ctx.saved_tensors
        need_mat, need_vec = ctx.needs_input_grad[:2]
        dev, cdt = _work_device(mat.device), D.compute_dtype(mat, vec)
        g = g.to(device=dev, dtype=cdt)
        d_mat = d_vec = None
        if need_mat:
            d_mat = _grad_for(dense_outer(g.unsqueeze(-1), vec.to(device=dev, dtype=cdt).unsqueeze(-1), False, False, 1), mat)
        if need_vec:
            d_vec = _grad_for(dense_tmatvec(mat.to(device=dev, dtype=cdt), g), vec)
        return d_mat, d_vec


def batchmatvec(mat, vec, out) -> Tensor:
    _check_out(out, "batchmatvec")
    return _BatchMatvec.apply(torch.as_tensor(mat), torch.as_tensor(vec))


class _Division(torch.autograd.Function):
    """X = A^-1 B (lmdiv, ``right`` False) or Y = B A^-1 (rmdiv: sugar.rmdiv(b, a) in its own names)."""

    @staticmethod
    def forward(ctx, a, b, method, right):
        from . import sugar
        res = sugar._rmdiv(b, a, method) if right else sugar._lmdiv(a, b, method)
        ctx.save_for_backward(a, res)
        ctx.right = right
        ctx.algo = sugar._algo(method)
        ctx.b = _meta(b)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        a, x = ctx.saved_tensors
        need_a, need_b = ctx.needs_input_grad[:2]
        dev, cdt = _work_device(a.device), x.dtype
        ac = a.to(device=dev, dtype=cdt)
        u = dense_tsolve(ac, g.to(device=dev, dtype=cdt), ctx.right, ctx.algo)
        d_a = d_b = None
        if need_b:
            d_b = _grad_for(u, ctx.b)
        if need_a:
            xc = x.to(device=dev)
            sym = ctx.algo == _lib.ALGO_LDL
            d = dense_outer(xc, u, True, sym, -1) if ctx.right else dense_outer(u, xc, False, sym, -1)
            d_a = _grad_for(d, a)
        return d_a, d_b, None, None


def lmdiv(a, b, method, out) -> Tensor:
    _check_out(out, "lmdiv")
    return _Division.apply(torch.as_tensor(a), torch.as_tensor(b), method, False)


def rmdiv(a, b, method, out) -> Tensor:
    """``a b^-1``: the Function's matrix is ``b``."""
    _check_out(out, "rmdiv")
    return _Division.apply(torch.as_tensor(b), torch.as_tensor(a), method, True)


# ---------------------------------------------------------------------------
# Gauss-Newton builders: sym_matmul, sym_outer, sym_to_full, sym_matmul_solve, sym_solve_update
# ---------------------------------------------------------------------------

def matmul_backward(j: Tensor, h: Tensor, g: Tensor, which: int):
    """(dJ, dH) of ``sym_matmul`` from J (..., k, d), packed H and the packed incoming gradient;
    ``which`` bit 0 asks for dJ, bit 1 for dH (None where not asked).  With both, one record
    [dJ | dH] per matrix is written and split into two views."""
    k, d = j.shape[-2:]
    kd, kk = k * d, h.shape[-1]
    batch = _batch((j, 2), (h, 1), (g, 1))
    out_len = (kd if which & 1 else 0) + (kk if which & 2 else 0)
    out = D.launch("nfm_sym_matmul_backward", (k, d, S._mode(k, d), which), batch, [(j.flatten(-2), 1), (h, 1), (g, 1)],
                   rec=(out_len,), dtype=h.dtype, device=h.device, skip_empty=True)
    return (out[..., :kd].unflatten(-1, (k, d)) if which & 1 else None,
            out[..., out_len - kk:] if which & 2 else None)


def outer_backward(x: Tensor, g: Tensor) -> Tensor:
    """Gradient of ``sym_outer``: 2 G^ x."""
    n = x.shape[-1]
    return D.launch("nfm_sym_outer_backward", (n,), _batch((x, 1), (g, 1)), [(x, 1), (g, 1)], rec=(n,), dtype=x.dtype,
                    device=x.device, skip_empty=True)


def to_full_backward(g: Tensor) -> Tensor:
    """Gradient of ``sym_to_full`` from the (..., n, n) incoming gradient: G_ii, G_ij + G_ji."""
    n = g.shape[-1]
    return D.launch("nfm_sym_to_full_backward", (n,), tuple(g.shape[:-2]), [(g.flatten(-2), 1)], rec=(n * (n + 1) // 2,),
                    dtype=g.dtype, device=g.device, skip_empty=True)


class _SymMatmul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, j, h):
        res = S._matmul(j, h)
        ctx.save_for_backward(j, h)
        ctx.cdt = res.dtype
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        j, h = ctx.saved_tensors
        need_j, need_h = ctx.needs_input_grad[:2]
        dev, cdt = _work_device(h.device), ctx.cdt
        dj, dh = matmul_backward(j.to(device=dev, dtype=cdt), h.to(device=dev, dtype=cdt), g.to(device=dev, dtype=cdt),
                                 int(need_j) | 2 * int(need_h))
        return _grad_for(dj, j), _grad_for(dh, h)


def matmul(j, h) -> Tensor:
    j, h = torch.as_tensor(j), torch.as_tensor(h)
    return _SymMatmul.apply(j, S._packed_h(j, h))


class _SymOuter(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return S._outer(x)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, = ctx.saved_tensors
        dev, cdt = _work_device(x.device), D.compute_dtype(x)
        return _grad_for(outer_backward(x.to(device=dev, dtype=cdt), g.to(device=dev, dtype=cdt)), x)


def outer(x) -> Tensor:
    return _SymOuter.apply(torch.as_tensor(x))


class _SymToFull(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p):
        ctx.p = _meta(p)
        return S._to_full(p)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        dev, cdt = _work_device(ctx.p.device), D.compute_dtype(g)
        return _grad_for(to_full_backward(g.to(device=dev, dtype=cdt)), ctx.p)


def to_full(p) -> Tensor:
    return _SymToFull.apply(torch.as_tensor(p))


class _MatmulSolve(torch.autograd.Function):
    """x = (A + diag d)^-1 g0 with A = sym_matmul(J, H).  Backward recomputes A (nfm_sym_matmul):
    u = (A + diag d)^-1 G (nfm_sym_solve, 'auto' as the fused kernel), dg0 = u, dA = -S(u, x),
    dd = -u * x (the diagonal of dA), and (dJ, dH) from dA by the sym_matmul backward."""

    @staticmethod
    def forward(ctx, j, h, g, diag):
        res = S._matmul_solve(j, h, g, diag)
        reg_t = diag if torch.is_tensor(diag) else None
        ctx.save_for_backward(j, h, res, reg_t)
        ctx.reg = None if reg_t is not None else diag   # float / sequence regulariser: no gradient
        ctx.g = _meta(g)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, gr):
        j, h, x, reg_t = ctx.saved_tensors
        need_j, need_h, need_g, need_d = ctx.needs_input_grad[:4]
        cdt, d = x.dtype, x.shape[-1]
        jc, hc = j.to(cdt), h.to(cdt)
        u = S._solve(S._matmul(jc, hc), gr.to(cdt), reg_t if reg_t is not None else ctx.reg, method="auto")
        d_j = d_h = d_g = d_d = None
        if need_g:
            d_g = _grad_for(u, ctx.g)
        if need_j or need_h:
            da = outer2(u, x, _lib.LAYOUT_SYM, -1)
            dj, dh = matmul_backward(jc, hc, da, int(need_j) | 2 * int(need_h))
            d_j, d_h = _grad_for(dj, j), _grad_for(dh, h)
            if need_d:
                d_d = _grad_for(da[..., :d], reg_t)
        elif need_d:
            d_d = _grad_for(outer2(u, x, _lib.LAYOUT_DIAG, -1), reg_t)
        return d_j, d_h, d_g, d_d


def matmul_solve(j, h, g, diag, out) -> Tensor:
    _check_out(out, "sym_matmul_solve")
    j, h, g = torch.as_tensor(j), torch.as_tensor(h), torch.as_tensor(g)
    return _MatmulSolve.apply(j, S._packed_h(j, h), g, diag)


class _SolveUpdate(torch.autograd.Function):
    """out = x - alpha s, s = (A + lam I + diag d)^-1 v.  Backward: dx = G; with
    u = (A + lam I + diag d)^-1 G and s recomputed (nfm_sym_solve, regulariser lam + d, the same
    method): dv = -alpha u, dp = alpha S(u, s), dd = alpha u * s (the diagonal of dp)."""

    @staticmethod
    def forward(ctx, x, mat, vec, diag, lam, alpha, method, inplace):
        res = S._solve_update(x, mat, vec, lam, alpha, x if inplace else None, diag=diag, method=method)
        if inplace:
            ctx.mark_dirty(x)
        reg_t = diag if torch.is_tensor(diag) else None
        ctx.save_for_backward(mat, vec, reg_t)
        ctx.reg = None if reg_t is not None else diag
        ctx.lam, ctx.alpha, ctx.method = float(lam), float(alpha), method
        ctx.cdt = D.compute_dtype(x, mat, vec)
        ctx.x = _meta(x)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        mat, vec, reg_t = ctx.saved_tensors
        need_x, need_m, need_v, need_d = ctx.needs_input_grad[:4]
        cdt, n = ctx.cdt, vec.shape[-1]
        d_x = d_m = d_v = d_d = None
        if need_x:
            d_x = _grad_for(g, ctx.x)
        if need_m or need_v or need_d:
            m = mat.to(cdt)
            reg = S._as_diag(reg_t if reg_t is not None else ctx.reg, n, cdt, m.device)
            reg = (ctx.lam or None) if reg is None else reg + ctx.lam
            ua = S._solve(m, g.to(cdt), reg, method=ctx.method) * ctx.alpha
            if need_v:
                d_v = _grad_for(-ua, vec)
            if need_m or need_d:
                s = S._solve(m, vec.to(cdt), reg, method=ctx.method)
                dp = outer2(ua, s, _lib.LAYOUT_SYM if need_m else _lib.LAYOUT_DIAG, 1)
                d_m = _grad_for(dp, mat) if need_m else None
                d_d = _grad_for(dp[..., :n], reg_t) if need_d else None
        return d_x, d_m, d_v, d_d, None, None, None, None


def solve_update(x, mat, vec, lam, alpha, out, diag, method, inplace: bool = False) -> Tensor:
    _check_out(out, "sym_solve_update")
    x, mat, vec = torch.as_tensor(x), torch.as_tensor(mat), torch.as_tensor(vec)
    return _SolveUpdate.apply(x, mat, vec, diag, lam, alpha, method, inplace)
