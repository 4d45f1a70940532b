"""Gradients of the Gauss-Newton builders: sym_matmul, sym_outer, sym_to_full, sym_matmul_solve
and sym_solve_update(_) (nitorch_fastmath_b200/_autograd.py, csrc/nfm_gn_grad.cu).

The formulas are written once here (``ref_*``) and pinned to autograd through the oracle on
CPU fp64; the GPU tests run ``torch.autograd.gradcheck`` and compare the library against
autograd through the oracle."""
import ctypes

import pytest
import torch

from conftest import TOL
from nitorch_fastmath_b200 import _lib
from oracle import generators as G
from oracle import ref_port as P

F64 = torch.float64
DTYPES = [torch.float32, torch.float64]
NS = list(range(1, 11))


# ---------------------------------------------------------------------------
# reference formulas (DESIGN.md section 8.2)
# ---------------------------------------------------------------------------

def _ghat(g):
    """Full symmetric form of a packed gradient with the off-diagonals halved."""
    f = P.sym_to_full(g)
    return 0.5 * (f + torch.diag_embed(torch.diagonal(f, 0, -2, -1)))


def _pack(m):
    """M_ii, 2 M_ij: the gradient with respect to p of <M, A(p)> for a symmetric M."""
    n = m.shape[-1]
    return torch.stack([m[..., i, j] if i == j else 2 * m[..., i, j] for i, j in P.packed_order(n)], -1)


def ref_S(u, w, layout="S"):
    if layout == "D":
        return u * w
    n = u.shape[-1]
    return torch.stack([u[..., i] * w[..., i] if i == j else u[..., i] * w[..., j] + u[..., j] * w[..., i]
                        for i, j in P.packed_order(n)], -1)


def jhj(j, h, mode):
    """Y = J^T H J (mode 0) or J H J^T (mode 1), packed, through torch."""
    hf = P.sym_to_full(h)
    full = j @ hf @ j.mT if mode == 1 else j.mT @ hf @ j
    return P.full_to_sym(full)


def mode_of(k, d):
    return 1 if (k == d and k <= 3) else 0


def ref_matmul(j, h, g, mode):
    """dJ, dH of jhj."""
    gh, hf = _ghat(g), P.sym_to_full(h)
    if mode == 0:
        return 2 * hf @ j @ gh, _pack(j @ gh @ j.mT)
    return 2 * gh @ j @ hf, _pack(j.mT @ gh @ j)


def ref_outer(x, g):
    return 2 * (_ghat(g) @ x.unsqueeze(-1)).squeeze(-1)


def ref_to_full(gf):
    n = gf.shape[-1]
    return torch.stack([gf[..., i, i] if i == j else gf[..., i, j] + gf[..., j, i] for i, j in P.packed_order(n)], -1)


def _solve(p, v, d):
    return torch.linalg.solve(P.sym_to_full(p) + torch.diag_embed(d), v.unsqueeze(-1)).squeeze(-1)


def ref_matmul_solve(j, h, g0, d, g, mode):
    """dJ, dH, dg0, dd of x = (jhj + diag d)^-1 g0."""
    a = jhj(j, h, mode)
    x, u = _solve(a, g0, d), _solve(a, g, d)
    da = -ref_S(u, x)
    dj, dh = ref_matmul(j, h, da, mode)
    return dj, dh, u, -u * x


def ref_solve_update(p, v, d, lam, alpha, g):
    """dx, dp, dv, dd of out = x - alpha (A + lam I + diag d)^-1 v."""
    s, u = _solve(p, v, d + lam), _solve(p, g, d + lam)
    return g, alpha * ref_S(u, s), -alpha * u, alpha * u * s


def _oracle_grads(fn, inputs, g):
    inputs = [t.detach().clone().requires_grad_() for t in inputs]
    return torch.autograd.grad(fn(*inputs), inputs, g)


def _close(a, b, tol=1e-10):
    return G.rel_err(a, b, 2 if a.dim() >= 3 else 1) < tol


def _jac(batch, k, d, dtype, seed, dev="cpu"):
    """A well-conditioned Jacobian: 0.1 randn plus ones on its leading diagonal (J^T H J + diag d stays
    well conditioned on every one of the parity batch's matrices, as the fp32 bar needs)."""
    j = G.vectors((batch, k), d, F64, seed=seed) * 0.1
    j[..., range(min(k, d)), range(min(k, d))] += 1.0
    return j.to(dtype).to(dev)


def _reg(batch, d, dtype, seed, dev="cpu"):
    return (1 + torch.rand(batch, d, dtype=F64, generator=G.gen(seed))).to(dtype).to(dev)


# ---------------------------------------------------------------------------
# CPU: the formulas against autograd through the oracle, fp64
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("d", NS)
@pytest.mark.parametrize("k", NS)
def test_matmul_formula_mode0(k, d):
    j, h, g = _jac(4, k, d, F64, k), G.spd_packed(4, k, F64, seed=d), G.vectors(4, d * (d + 1) // 2, F64, seed=3)
    fn = (lambda j, h: jhj(j, h, 0)) if mode_of(k, d) == 1 else P.sym_matmul   # the oracle's own J^T H J branch
    gj, gh = _oracle_grads(fn, [j, h], g)
    dj, dh = ref_matmul(j, h, g, 0)
    assert _close(gj, dj) and _close(gh, dh)


@pytest.mark.parametrize("n", [1, 2, 3])
def test_matmul_formula_mode1(n):
    j, h, g = _jac(4, n, n, F64, n), G.spd_packed(4, n, F64, seed=n), G.vectors(4, n * (n + 1) // 2, F64, seed=3)
    gj, gh = _oracle_grads(P.sym_matmul, [j, h], g)
    dj, dh = ref_matmul(j, h, g, 1)
    assert _close(gj, dj) and _close(gh, dh)


@pytest.mark.parametrize("k,d", [(2, 2), (3, 3), (4, 2), (6, 6), (10, 3), (8, 5)])
def test_matmul_formula_diagonal_h(k, d):
    """A diagonal H is padded to packed form outside the Function: its gradient is the diagonal of dH."""
    mode = mode_of(k, d)
    j, hd, g = _jac(4, k, d, F64, 1), 1 + torch.rand(4, k, dtype=F64, generator=G.gen(2)), G.vectors(4, d * (d + 1) // 2, F64, seed=3)
    pad = lambda h: torch.cat([h, h.new_zeros(*h.shape[:-1], k * (k - 1) // 2)], -1)   # noqa: E731
    gj, gh = _oracle_grads(lambda j, h: P.sym_matmul(j, pad(h)), [j, hd], g)
    dj, dh = ref_matmul(j, pad(hd), g, mode)
    assert _close(gj, dj) and _close(gh, dh[..., :k])


@pytest.mark.parametrize("n", NS)
def test_outer_and_to_full_formulas(n):
    x, g = G.vectors(5, n, F64, seed=1), G.vectors(5, n * (n + 1) // 2, F64, seed=2)
    gx, = _oracle_grads(P.sym_outer, [x], g)
    assert _close(gx, ref_outer(x, g))
    p, gf = G.spd_packed(5, n, F64, seed=n), G.vectors((5, n), n, F64, seed=3)
    gp, = _oracle_grads(P.sym_to_full, [p], gf)
    assert _close(gp, ref_to_full(gf))


@pytest.mark.parametrize("k,d", [(1, 1), (2, 2), (3, 3), (1, 4), (4, 2), (6, 6), (5, 6), (10, 3), (7, 1)])
def test_matmul_solve_formula(k, d):
    mode = mode_of(k, d)
    j, h, g0 = _jac(4, k, d, F64, 1), G.spd_packed(4, k if mode == 0 else d, F64, seed=2), G.vectors(4, d, F64, seed=3)
    dd, g = _reg(4, d, F64, 4), G.vectors(4, d, F64, seed=5)
    got = _oracle_grads(lambda j, h, g0, dd: P.sym_solve(P.sym_matmul(j, h), g0, dd), [j, h, g0, dd], g)
    assert all(_close(a, b) for a, b in zip(got, ref_matmul_solve(j, h, g0, dd, g, mode)))


@pytest.mark.parametrize("n", NS)
def test_solve_update_formula(n):
    x, p, v = G.vectors(4, n, F64, seed=1), G.spd_packed(4, n, F64, seed=n), G.vectors(4, n, F64, seed=2)
    dd, g = _reg(4, n, F64, 3), G.vectors(4, n, F64, seed=4)
    lam, alpha = 0.25, 0.7
    got = _oracle_grads(lambda x, p, v, dd: x - alpha * P.sym_solve(p, v, dd + lam), [x, p, v, dd], g)
    assert all(_close(a, b) for a, b in zip(got, ref_solve_update(p, v, dd, lam, alpha, g)))


def test_gn_backward_entry_points_reject_bad_arguments_without_a_gpu():
    lib = _lib.load()
    buf = ctypes.create_string_buffer(4096)
    q = ctypes.addressof(buf)
    F32 = _lib.F32
    mm = lib.nfm_sym_matmul_backward
    # nfm_sym_matmul_backward(dtype, k, d, mode, which, batch, jac, js, hess, hs, grad, gs, out, os, stream)
    for k, d, mode in [(3, 3, 1), (6, 6, 0), (10, 3, 0), (8, 5, 0), (10, 10, 0), (5, 5, 1)]:   # register and run-time kernels
        js, hs, gs = k * d, (k if mode == 0 else d) * ((k if mode == 0 else d) + 1) // 2, (d if mode == 0 else k) * ((d if mode == 0 else k) + 1) // 2
        os_ = js + hs
        assert mm(7, k, d, mode, 3, 4, q, js, q, hs, q, gs, q, os_, None) == -1
        assert mm(F32, k, d, 2, 3, 4, q, js, q, hs, q, gs, q, os_, None) == -1
        assert mm(F32, k, d, mode, 0, 4, q, js, q, hs, q, gs, q, os_, None) == -1
        assert mm(F32, k, d, mode, 4, 4, q, js, q, hs, q, gs, q, os_, None) == -1
        assert mm(F32, k, d, mode, 3, 4, None, js, q, hs, q, gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, None, hs, q, gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, q, hs, None, gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, q, hs, q, gs, None, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, -js, q, hs, q, gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, q, -hs, q, gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, q, hs, q, -gs, q, os_, None) == -2
        assert mm(F32, k, d, mode, 3, 4, q, js, q, hs, q, gs, q, -os_, None) == -2
        assert mm(F32, k, d, mode, 3, -4, q, js, q, hs, q, gs, q, os_, None) == -2
        for which in (1, 2, 3):
            assert mm(F32, k, d, mode, which, 0, q, js, q, hs, q, gs, q, os_, None) == 0
    assert mm(F32, 0, 3, 0, 3, 4, q, 0, q, 0, q, 6, q, 6, None) == -1
    assert mm(F32, 11, 3, 0, 3, 4, q, 33, q, 66, q, 6, q, 99, None) == -1
    assert mm(F32, 3, 11, 0, 3, 4, q, 33, q, 6, q, 66, q, 39, None) == -1
    assert mm(F32, 3, 2, 1, 3, 4, q, 6, q, 3, q, 6, q, 9, None) == -1      # mode 1 needs k == d
    assert b"k == d" in lib.nfm_last_error_string()
    # nfm_sym_outer_backward(dtype, n, batch, vec, vs, grad, gs, out, os, stream)
    ob = lib.nfm_sym_outer_backward
    assert ob(7, 3, 4, q, 3, q, 6, q, 3, None) == -1
    assert ob(F32, 0, 4, q, 0, q, 0, q, 0, None) == -1
    assert ob(F32, 11, 4, q, 11, q, 66, q, 11, None) == -1
    assert ob(F32, 3, 4, None, 3, q, 6, q, 3, None) == -2
    assert ob(F32, 3, 4, q, 3, None, 6, q, 3, None) == -2
    assert ob(F32, 3, 4, q, 3, q, 6, None, 3, None) == -2
    assert ob(F32, 3, 4, q, -3, q, 6, q, 3, None) == -2
    assert ob(F32, 3, 4, q, 3, q, -6, q, 3, None) == -2
    assert ob(F32, 3, 4, q, 3, q, 6, q, -3, None) == -2
    assert ob(F32, 3, -4, q, 3, q, 6, q, 3, None) == -2
    assert ob(F32, 3, 0, q, 3, q, 6, q, 3, None) == 0
    # nfm_sym_to_full_backward(dtype, n, batch, grad, gs, out, os, stream)
    tb = lib.nfm_sym_to_full_backward
    assert tb(7, 3, 4, q, 9, q, 6, None) == -1
    assert tb(F32, 0, 4, q, 0, q, 0, None) == -1
    assert tb(F32, 11, 4, q, 121, q, 66, None) == -1
    assert tb(F32, 3, 4, None, 9, q, 6, None) == -2
    assert tb(F32, 3, 4, q, 9, None, 6, None) == -2
    assert tb(F32, 3, 4, q, -9, q, 6, None) == -2
    assert tb(F32, 3, 4, q, 9, q, -6, None) == -2
    assert tb(F32, 3, -4, q, 9, q, 6, None) == -2
    assert tb(F32, 3, 0, q, 9, q, 6, None) == 0


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------

@pytest.fixture(scope="module")
def nfm():
    import nitorch_fastmath_b200 as m
    return m


def _leaf(t):
    return t.detach().clone().requires_grad_()


def _gradcheck(fn, *inputs):
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-7, rtol=1e-5)


def _grads(fn, inputs, g):
    leaves = [_leaf(t) for t in inputs]
    return torch.autograd.grad(fn(*leaves), leaves, g)


MM_SHAPES = [(1, 1), (2, 2), (3, 3), (4, 2), (2, 5), (6, 6), (10, 3), (8, 5), (10, 10), (4, 8)]   # (8, 5) on: run-time kernel


@pytest.mark.gpu
@pytest.mark.parametrize("k,d", MM_SHAPES)
def test_gradcheck_matmul(nfm, k, d):
    kh = k if mode_of(k, d) == 0 else d
    j, h = _leaf(_jac(2, k, d, F64, 1, "cuda")), _leaf(G.spd_packed(2, kh, F64, seed=2).cuda())
    _gradcheck(nfm.sym_matmul, j, h)
    _gradcheck(nfm.sym_matmul, j, _leaf(1 + torch.rand(2, kh, dtype=F64, device="cuda")))       # diagonal h
    _gradcheck(nfm.sym_matmul, j, _leaf(h.detach()[0]))                                         # broadcast h (kk,)
    _gradcheck(nfm.sym_matmul, _leaf(j.detach()[0]), h)                                         # broadcast J
    _gradcheck(lambda j: nfm.sym_matmul(j, h.detach()), j)                                      # dJ only
    _gradcheck(lambda h: nfm.sym_matmul(j.detach(), h), h)                                      # dH only


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
def test_gradcheck_outer_and_to_full(nfm, n):
    _gradcheck(nfm.sym_outer, _leaf(G.vectors(3, n, F64, seed=1).cuda()))
    _gradcheck(nfm.sym_to_full, _leaf(G.spd_packed(3, n, F64, seed=2).cuda()))


@pytest.mark.gpu
@pytest.mark.parametrize("k,d", [(1, 1), (2, 2), (3, 3), (4, 2), (2, 5), (6, 6), (10, 3), (7, 1)])
def test_gradcheck_matmul_solve(nfm, k, d):
    kh = k if mode_of(k, d) == 0 else d
    j, h = _leaf(_jac(2, k, d, F64, 1, "cuda")), _leaf(G.spd_packed(2, kh, F64, seed=2).cuda())
    g0, dd = _leaf(G.vectors(2, d, F64, seed=3).cuda()), _leaf(_reg(2, d, F64, 4, "cuda"))
    _gradcheck(nfm.sym_matmul_solve, j, h, g0, dd)                                               # tensor regulariser
    _gradcheck(lambda j, h, g0: nfm.sym_matmul_solve(j, h, g0, 1.5), j, h, g0)                   # float regulariser
    _gradcheck(lambda j, h, g0: nfm.sym_matmul_solve(j, h, g0, [1.0, 2.0][:d]), j, h, g0)        # sequence
    _gradcheck(lambda h, dd: nfm.sym_matmul_solve(j.detach(), h, g0.detach(), dd),
               _leaf(1 + torch.rand(2, kh, dtype=F64, device="cuda")), dd)                         # diagonal h
    _gradcheck(lambda h: nfm.sym_matmul_solve(j.detach(), h, g0.detach(), dd.detach()), _leaf(h.detach()[0]))  # broadcast h
    _gradcheck(lambda dd: nfm.sym_matmul_solve(j.detach(), h.detach(), g0.detach(), dd), _leaf(dd.detach()[0]))  # 1-D regulariser


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["auto", "ldl"])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_solve_update(nfm, n, method):
    x, p, v = _leaf(G.vectors(2, n, F64, seed=1).cuda()), _leaf(G.spd_packed(2, n, F64, seed=n).cuda()), _leaf(G.vectors(2, n, F64, seed=2).cuda())
    dd = _leaf(_reg(2, n, F64, 3, "cuda"))
    _gradcheck(lambda x, p, v, dd: nfm.sym_solve_update(x, p, v, 0.3, 0.7, diag=dd, method=method), x, p, v, dd)
    _gradcheck(lambda x, p, v: nfm.sym_solve_update(x, p, v, method=method), x, p, v)
    _gradcheck(lambda x, p, v, dd: nfm.sym_solve_update_(x.clone(), p, v, 0.3, 0.7, diag=dd, method=method), x, p, v, dd)
    _gradcheck(lambda p: nfm.sym_solve_update(x.detach(), p, v.detach(), 0.1, 2.0, method=method), _leaf(p.detach()[0]))


BIG = 65536 + 37          # full TMA tiles, a partial tile and a strided tail; ragged
PARITY = [("matmul", 3, 3), ("matmul", 6, 6), ("matmul", 10, 3), ("matmul", 4, 2), ("matmul", 8, 5),
          ("matmul_solve", 3, 3), ("matmul_solve", 6, 6), ("matmul_solve", 10, 3),
          ("solve_update", 3, 0), ("solve_update", 6, 0), ("solve_update", 10, 0),
          ("outer", 3, 0), ("outer", 10, 0), ("to_full", 6, 0), ("to_full", 10, 0)]


def _parity_case(kind, k, d, dtype):
    """Inputs in ``dtype``, the incoming gradient, the library call and the fp64 oracle chain."""
    if kind in ("matmul", "matmul_solve"):
        kh = k if mode_of(k, d) == 0 else d
        ins = [_jac(BIG, k, d, dtype, 1), G.spd_packed(BIG, kh, dtype, seed=2)]
        if kind == "matmul":
            return ins, G.vectors(BIG, d * (d + 1) // 2 if mode_of(k, d) == 0 else k * (k + 1) // 2, dtype, seed=5), "sym_matmul", P.sym_matmul
        ins += [G.vectors(BIG, d, dtype, seed=3), _reg(BIG, d, dtype, 4)]
        return ins, G.vectors(BIG, d, dtype, seed=5), "sym_matmul_solve", lambda j, h, g0, dd: P.sym_solve(P.sym_matmul(j, h), g0, dd)
    n = k
    if kind == "solve_update":
        ins = [G.vectors(BIG, n, dtype, seed=1), G.spd_packed(BIG, n, dtype, seed=2), G.vectors(BIG, n, dtype, seed=3), _reg(BIG, n, dtype, 4)]
        return (ins, G.vectors(BIG, n, dtype, seed=5), lambda nfm: lambda x, p, v, dd: nfm.sym_solve_update(x, p, v, 0.5, 0.8, diag=dd),
                lambda x, p, v, dd: x - 0.8 * P.sym_solve(p, v, dd + 0.5))
    if kind == "outer":
        return [G.vectors(BIG, n, dtype, seed=1)], G.vectors(BIG, n * (n + 1) // 2, dtype, seed=5), "sym_outer", P.sym_outer
    return [G.spd_packed(BIG, n, dtype, seed=1)], G.vectors((BIG, n), n, dtype, seed=5), "sym_to_full", P.sym_to_full


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind,k,d", PARITY)
def test_gradient_parity_at_the_bars(nfm, kind, k, d, dtype):
    ins, g, call, oracle = _parity_case(kind, k, d, dtype)
    fn = getattr(nfm, call) if isinstance(call, str) else call(nfm)
    leaves = [_leaf(t.cuda()) for t in ins]
    got = torch.autograd.grad(fn(*leaves), leaves, g.cuda())
    ref = _oracle_grads(oracle, [t.to(F64) for t in ins], g.to(F64))
    for a, b in zip(got, ref):
        assert a.dtype == dtype and a.shape == b.shape
        err = G.rel_err(a, b, 2 if b.dim() == 3 else 1)
        assert err < TOL[dtype], (kind, k, d, dtype, err)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_new_kernels_take_the_tma_path_on_dense_aligned_fields(nfm, dtype):
    from nitorch_fastmath_b200 import _autograd as A
    lib = _lib.load()
    B = 8192
    for k, d in [(1, 1), (3, 3), (6, 6), (10, 3), (4, 2)]:
        mode = mode_of(k, d)
        kh, ko = (k, d) if mode == 0 else (d, k)
        j, h, g = _jac(B, k, d, dtype, 1, "cuda"), G.spd_packed(B, kh, dtype, seed=2).cuda(), G.vectors(B, ko * (ko + 1) // 2, dtype, seed=3).cuda()
        for which in (1, 2, 3):
            A.matmul_backward(j, h, g, which)
            assert lib.nfm_last_path_was_tma() == 1, (k, d, which)
    for n in (1, 3, 6, 10):
        A.outer_backward(G.vectors(B, n, dtype, seed=1).cuda(), G.vectors(B, n * (n + 1) // 2, dtype, seed=2).cuda())
        assert lib.nfm_last_path_was_tma() == 1
        A.to_full_backward(G.vectors((B, n), n, dtype, seed=3).cuda())
        assert lib.nfm_last_path_was_tma() == 1
    # the run-time-sized kernel for the shapes the forward runs there
    A.matmul_backward(_jac(B, 8, 5, dtype, 1, "cuda"), G.spd_packed(B, 8, dtype, seed=2).cuda(), G.vectors(B, 15, dtype, seed=3).cuda(), 3)
    assert lib.nfm_last_path_was_tma() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("k,d", [(3, 3), (6, 6), (10, 3), (8, 5)])
def test_views_give_the_bits_of_the_dense_call(nfm, k, d):
    """A head-peeled view (``field[1:]``, not 16-byte aligned) and a strided view (every other
    matrix) give the same gradient bits as the dense call on copies."""
    B = 4099
    kh = k if mode_of(k, d) == 0 else d
    ko = d if mode_of(k, d) == 0 else k
    j, h = _jac(B, k, d, torch.float32, 1, "cuda"), G.spd_packed(B, kh, torch.float32, seed=2).cuda()
    g = G.vectors(B, ko * (ko + 1) // 2, torch.float32, seed=3).cuda()
    x, gx = G.vectors(B, ko, torch.float32, seed=4).cuda(), G.vectors(B, ko * (ko + 1) // 2, torch.float32, seed=5).cuda()
    p, gf = G.spd_packed(B, ko, torch.float32, seed=6).cuda(), G.vectors((B, ko), ko, torch.float32, seed=7).cuda()
    cases = [(nfm.sym_matmul, [j, h], g), (nfm.sym_outer, [x], gx), (nfm.sym_to_full, [p], gf)]
    for fn, ins, gg in cases:
        for sl in (slice(1, None), slice(None, None, 2)):
            bases = [_leaf(t) for t in ins]
            views = [b[sl] for b in bases]
            got = torch.autograd.grad(fn(*views), views, gg[sl])
            ref = _grads(fn, [t[sl].contiguous() for t in ins], gg[sl].contiguous())
            assert all(torch.equal(a, b) for a, b in zip(got, ref)), (fn, sl)


@pytest.mark.gpu
def test_gradient_path_forward_and_no_grad_calls_are_unchanged(nfm):
    B = 4096
    f32 = torch.float32
    j, h, g0 = _jac(B, 3, 3, f32, 1, "cuda"), G.spd_packed(B, 3, f32, seed=2).cuda(), G.vectors(B, 3, f32, seed=3).cuda()
    j6, h6, g6 = _jac(B, 6, 6, f32, 1, "cuda"), G.spd_packed(B, 6, f32, seed=2).cuda(), G.vectors(B, 6, f32, seed=3).cuda()
    x, dd = G.vectors(B, 6, f32, seed=4).cuda(), _reg(B, 6, f32, 5, "cuda")
    calls = [lambda a: nfm.sym_matmul(a[0], a[1]), lambda a: nfm.sym_matmul(a[3], a[4]), lambda a: nfm.sym_outer(a[2]),
             lambda a: nfm.sym_to_full(a[1]), lambda a: nfm.sym_matmul_solve(a[0], a[1], a[2], 1.0),
             lambda a: nfm.sym_matmul_solve(a[3], a[4], a[5], a[7]), lambda a: nfm.sym_solve_update(a[6], a[4], a[5], 0.1, 0.5),
             lambda a: nfm.sym_solve_update(a[6], a[4], a[5], 0.1, 0.5, diag=a[7])]
    base = [j, h, g0, j6, h6, g6, x, dd]
    for call in calls:
        b0 = _lib.launch_count()
        plain = call(base)
        d_plain = _lib.launch_count() - b0
        assert d_plain == 1
        leaves = [_leaf(t) for t in base]
        with torch.no_grad():
            b0 = _lib.launch_count()
            gated = call(leaves)
            d_gated = _lib.launch_count() - b0
        assert not gated.requires_grad and torch.equal(plain, gated) and d_gated == 1
        with_grad = call(leaves)
        assert with_grad.requires_grad and torch.equal(plain, with_grad.detach())
    # the in-place variant: same bits on a non-leaf
    xg = _leaf(x)
    y = nfm.sym_solve_update_(xg.clone(), _leaf(h6), g6, 0.1, 0.5)
    assert y.requires_grad and torch.equal(y.detach(), nfm.sym_solve_update(x, h6, g6, 0.1, 0.5))


@pytest.mark.gpu
def test_out_and_second_order_raise(nfm):
    j, h, g0 = _leaf(_jac(4, 3, 3, F64, 1, "cuda")), _leaf(G.spd_packed(4, 3, F64, seed=2).cuda()), _leaf(G.vectors(4, 3, F64, seed=3).cuda())
    x = _leaf(G.vectors(4, 3, F64, seed=4).cuda())
    with pytest.raises(RuntimeError):
        nfm.sym_matmul_solve(j, h, g0, out=torch.empty(4, 3, dtype=F64, device="cuda"))
    with pytest.raises(RuntimeError):
        nfm.sym_solve_update(x, h, g0, out=torch.empty(4, 3, dtype=F64, device="cuda"))
    for fn, leaf in [(lambda: nfm.sym_matmul(j, h), j), (lambda: nfm.sym_outer(x), x), (lambda: nfm.sym_to_full(h), h),
                     (lambda: nfm.sym_matmul_solve(j, h, g0), h), (lambda: nfm.sym_solve_update(x, h, g0, 0.1), h)]:
        ga, = torch.autograd.grad(fn().sum(), leaf, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(ga.sum(), leaf)


@pytest.mark.gpu
@pytest.mark.parametrize("k,d", [(3, 3), (6, 4), (8, 5)])
def test_cpu_operands_get_the_gradients_of_cuda_operands(nfm, k, d):
    kh = k if mode_of(k, d) == 0 else d
    ko = d if mode_of(k, d) == 0 else k
    j, h = _jac(64, k, d, F64, 1), G.spd_packed(64, kh, F64, seed=2)
    g, x, gx = G.vectors(64, ko * (ko + 1) // 2, F64, seed=3), G.vectors(64, ko, F64, seed=4), G.vectors(64, ko * (ko + 1) // 2, F64, seed=5)
    gf = G.vectors((64, kh), kh, F64, seed=6)
    for fn, ins, gg in [(nfm.sym_matmul, [j, h], g), (nfm.sym_outer, [x], gx), (nfm.sym_to_full, [h], gf)]:
        got = _grads(fn, ins, gg)
        ref = _grads(fn, [t.cuda() for t in ins], gg.cuda())
        assert all(a.device.type == "cpu" and _close(a, b, 1e-12) for a, b in zip(got, ref))


@pytest.mark.gpu
def test_mixed_and_half_dtypes_return_gradients_in_the_input_dtypes(nfm):
    j, h = _leaf(_jac(32, 6, 3, F64, 1, "cuda")), _leaf(G.spd_packed(32, 6, torch.float32, seed=2).cuda())
    gj, gh = torch.autograd.grad(nfm.sym_matmul(j, h).sum(), (j, h))
    assert gj.dtype == F64 and gh.dtype == torch.float32
    x, p, v = (_leaf(G.vectors(32, 3, torch.float32, seed=1).cuda()), _leaf(G.spd_packed(32, 3, F64, seed=2).cuda()),
               _leaf(G.vectors(32, 3, torch.float32, seed=3).cuda()))
    grads = torch.autograd.grad(nfm.sym_solve_update(x, p, v, 0.1).sum(), (x, p, v))
    assert [t.dtype for t in grads] == [torch.float32, F64, torch.float32]
    xh = _leaf(G.vectors(32, 4, torch.half, seed=4).cuda())
    gx, = torch.autograd.grad(nfm.sym_outer(xh).float().sum(), xh)
    assert gx.dtype == torch.half
    ref, = _grads(nfm.sym_outer, [xh.detach().float()], torch.ones(32, 10, device="cuda"))
    assert _close(gx.float(), ref, 1e-3)
    ph = _leaf(G.spd_packed(32, 4, torch.bfloat16, seed=5).cuda())
    gp, = torch.autograd.grad(nfm.sym_to_full(ph).float().sum(), ph)
    assert gp.dtype == torch.bfloat16
    jh, hh = _leaf(_jac(32, 4, 2, torch.half, 1, "cuda")), _leaf(G.spd_packed(32, 4, torch.half, seed=6).cuda())
    gj, gh = torch.autograd.grad(nfm.sym_matmul(jh, hh).float().sum(), (jh, hh))
    assert gj.dtype == torch.half and gh.dtype == torch.half


@pytest.mark.gpu
def test_registration_chain_gets_every_gradient(nfm):
    """H = sym_matmul(J, h) -> sym_solve(H, g): the gradients reach J and h, and agree with the
    fused sym_matmul_solve and with the oracle."""
    B, k, d = 512, 6, 3
    j, h, g = _jac(B, k, d, F64, 1, "cuda"), G.spd_packed(B, k, F64, seed=2).cuda(), G.vectors(B, d, F64, seed=3).cuda()
    w = G.vectors(B, d, F64, seed=4).cuda()
    chain = _grads(lambda j, h, g: nfm.sym_solve(nfm.sym_matmul(j, h), g, 1.0), [j, h, g], w)
    fused = _grads(lambda j, h, g: nfm.sym_matmul_solve(j, h, g, 1.0), [j, h, g], w)
    ref = _oracle_grads(lambda j, h, g: P.sym_solve(P.sym_matmul(j, h), g, 1.0), [t.cpu() for t in (j, h, g)], w.cpu())
    for a, b, c in zip(chain, fused, ref):
        assert _close(a, c, 1e-12) and _close(b, c, 1e-12)
