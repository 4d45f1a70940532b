"""Gradients of sym_matvec / sym_addmatvec / sym_submatvec, sym_solve, sym_invert
and sym_det (nitorch_fastmath_b200/_autograd.py, csrc/nfm_sym_grad.cu).

The formulas are written once here (``ref_*``) and pinned to autograd through
the oracle on CPU fp64; the GPU tests compare the library against autograd
through the oracle and run ``torch.autograd.gradcheck``."""
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
LAYOUTS = {"E": _lib.LAYOUT_SCALED_IDENTITY, "D": _lib.LAYOUT_DIAG, "S": _lib.LAYOUT_SYM}


# ---------------------------------------------------------------------------
# reference formulas (DESIGN.md, "Gradients")
# ---------------------------------------------------------------------------

def ref_S(u, w, layout="S"):
    """Gradient of u^T A w with respect to the stored coefficients of A."""
    n = u.shape[-1]
    if layout == "E":
        return (u * w).sum(-1, keepdim=True)
    if layout == "D":
        return u * w
    return torch.stack([u[..., i] * w[..., i] if i == j else u[..., i] * w[..., j] + u[..., j] * w[..., i]
                        for i, j in P.packed_order(n)], -1)


def _pack_sym_grad(m):
    """Gradient with respect to p of <M, A(p)> for a symmetric M: M_ii, 2 M_ij."""
    n = m.shape[-1]
    return torch.stack([m[..., i, j] if i == j else 2 * m[..., i, j] for i, j in P.packed_order(n)], -1)


def ref_matvec(p, v, g, sign):
    """d_v, d_p of y = inp + sign * A v (sign 0: y = A v)."""
    s = -1.0 if sign < 0 else 1.0
    a = P.sym_to_full(p)
    return s * (a @ g.unsqueeze(-1)).squeeze(-1), s * ref_S(g, v)


def ref_solve(p, v, d, g):
    """d_p, d_v, d_d of x = (A + diag d)^-1 v."""
    a = P.sym_to_full(p) + torch.diag_embed(d)
    x = torch.linalg.solve(a, v)
    u = torch.linalg.solve(a, g)
    return -ref_S(u, x), u, -u * x


def ref_invert(p, g, diag):
    b = torch.linalg.inv(P.sym_to_full(p))
    n = b.shape[-1]
    if diag:
        gh = torch.diag_embed(g)
    else:
        gf = P.sym_to_full(g)
        gh = 0.5 * (gf + torch.diag_embed(torch.diagonal(gf, 0, -2, -1)))
    return -_pack_sym_grad(b @ gh @ b)


def ref_det(p, g):
    a = P.sym_to_full(p)
    return _pack_sym_grad((g * torch.det(a))[..., None, None] * torch.linalg.inv(a))


def _oracle_grads(fn, inputs, g):
    inputs = [t.detach().clone().requires_grad_() for t in inputs]
    out = fn(*inputs)
    return torch.autograd.grad(out, inputs, g)


def _close(a, b, tol=1e-12):
    return G.rel_err(a, b) < tol


# ---------------------------------------------------------------------------
# CPU: the formulas against autograd through the oracle
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("sign", [0, 1, -1])
def test_matvec_formula(n, sign):
    p, v, i0 = G.spd_packed(5, n, F64, seed=n), G.vectors(5, n, F64, seed=1), G.vectors(5, n, F64, seed=2)
    g = G.vectors(5, n, F64, seed=3)
    fn = {0: lambda i, p, v: P.sym_matvec(p, v) + 0 * i, 1: lambda i, p, v: P.sym_addmatvec(i, p, v),
          -1: lambda i, p, v: P.sym_submatvec(i, p, v)}[sign]
    gi, gp, gv = _oracle_grads(fn, [i0, p, v], g)
    dv, dp = ref_matvec(p, v, g, sign)
    assert _close(gp, dp) and _close(gv, dv) and (sign == 0 or _close(gi, g))


@pytest.mark.parametrize("n", NS)
def test_solve_formula(n):
    p, v, g = G.spd_packed(5, n, F64, seed=n), G.vectors(5, n, F64, seed=1), G.vectors(5, n, F64, seed=3)
    d = torch.rand(5, n, dtype=F64, generator=G.gen(4))
    gp, gv, gd = _oracle_grads(lambda p, v, d: P.sym_solve(p, v, d), [p, v, d], g)
    dp, dv, dd = ref_solve(p, v, d, g)
    assert _close(gp, dp, 1e-10) and _close(gv, dv, 1e-10) and _close(gd, dd, 1e-10)


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("diag", [False, True])
def test_invert_formula(n, diag):
    p = G.spd_packed(5, n, F64, seed=n)
    g = G.vectors(5, n if diag else n * (n + 1) // 2, F64, seed=3)
    gp, = _oracle_grads(lambda p: P.sym_invert(p, diag), [p], g)
    assert _close(gp, ref_invert(p, g, diag), 1e-10)


@pytest.mark.parametrize("n", NS)
def test_det_formula(n):
    p = G.spd_packed(5, n, F64, seed=n) / n        # keep the determinants O(1)
    g = torch.randn(5, dtype=F64, generator=G.gen(3))
    gp, = _oracle_grads(lambda p: torch.det(P.sym_to_full(p)), [p], g)
    assert _close(gp, ref_det(p, g), 1e-10)


def test_backward_entry_points_reject_bad_arguments_without_a_gpu():
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1024)
    q = ctypes.addressof(buf)
    F32, SYM = _lib.F32, _lib.LAYOUT_SYM
    # nfm_sym_outer2(dtype, n, layout, batch, u, us, w, ws, sign, out, os, stream)
    assert lib.nfm_sym_outer2(F32, 11, SYM, 4, q, 11, q, 11, 1, q, 66, None) == -1
    assert lib.nfm_sym_outer2(F32, 0, SYM, 4, q, 1, q, 1, 1, q, 1, None) == -1
    assert lib.nfm_sym_outer2(7, 3, SYM, 4, q, 3, q, 3, 1, q, 6, None) == -1
    assert lib.nfm_sym_outer2(F32, 3, _lib.LAYOUT_FULL, 4, q, 3, q, 3, 1, q, 9, None) == -1
    assert lib.nfm_sym_outer2(F32, 3, -1, 4, q, 3, q, 3, 1, q, 1, None) == -1
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, q, 3, q, 3, 0, q, 6, None) == -2
    assert b"sign" in lib.nfm_last_error_string()
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, None, 3, q, 3, 1, q, 6, None) == -2
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, q, 3, None, 3, 1, q, 6, None) == -2
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, q, 3, q, 3, 1, None, 6, None) == -2
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, q, -3, q, 3, 1, q, 6, None) == -2
    assert lib.nfm_sym_outer2(F32, 3, SYM, 4, q, 3, q, 3, 1, q, -6, None) == -2
    assert lib.nfm_sym_outer2(F32, 3, SYM, -1, q, 3, q, 3, 1, q, 6, None) == -2
    # nfm_sym_invert_backward(dtype, n, diag_only, batch, inv, is, grad, gs, out, os, stream)
    assert lib.nfm_sym_invert_backward(F32, 11, 0, 4, q, 66, q, 66, q, 66, None) == -1
    assert lib.nfm_sym_invert_backward(7, 3, 0, 4, q, 6, q, 6, q, 6, None) == -1
    assert lib.nfm_sym_invert_backward(F32, 3, 0, 4, None, 6, q, 6, q, 6, None) == -2
    assert lib.nfm_sym_invert_backward(F32, 3, 1, 4, q, 6, None, 3, q, 6, None) == -2
    assert lib.nfm_sym_invert_backward(F32, 3, 0, 4, q, 6, q, 6, None, 6, None) == -2
    assert lib.nfm_sym_invert_backward(F32, 3, 0, 4, q, 6, q, -6, q, 6, None) == -2
    assert lib.nfm_sym_invert_backward(F32, 3, 0, -4, q, 6, q, 6, q, 6, None) == -2
    # nfm_sym_det_backward(dtype, n, batch, mat, ms, grad, gs, out, os, stream)
    assert lib.nfm_sym_det_backward(F32, 11, 4, q, 66, q, 1, q, 66, None) == -1
    assert lib.nfm_sym_det_backward(7, 3, 4, q, 6, q, 1, q, 6, None) == -1
    assert lib.nfm_sym_det_backward(F32, 3, 4, None, 6, q, 1, q, 6, None) == -2
    assert lib.nfm_sym_det_backward(F32, 3, 4, q, 6, None, 1, q, 6, None) == -2
    assert lib.nfm_sym_det_backward(F32, 3, 4, q, 6, q, 1, None, 6, None) == -2
    assert lib.nfm_sym_det_backward(F32, 3, 4, q, -6, q, 1, q, 6, None) == -2
    assert lib.nfm_sym_det_backward(F32, 3, -4, q, 6, q, 1, q, 6, None) == -2
    # an empty batch is a no-op that touches nothing
    assert lib.nfm_sym_det_backward(F32, 3, 0, q, 6, q, 1, q, 6, None) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_gradient_path_fails_loudly_without_cuda():
    import nitorch_fastmath_b200 as nfm
    m = (torch.rand(8, 6) + 3).requires_grad_()
    v = torch.rand(8, 3).requires_grad_()
    calls = [lambda: nfm.sym_solve(m, v), lambda: nfm.sym_matvec(m, v), lambda: nfm.sym_addmatvec(v, m, v),
             lambda: nfm.sym_submatvec(v, m, v), lambda: nfm.sym_invert(m), lambda: nfm.sym_invert(m, True),
             lambda: nfm.sym_det(m)]
    for call in calls:
        with pytest.raises(RuntimeError):
            call()


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------

@pytest.fixture(scope="module")
def nfm():
    import nitorch_fastmath_b200 as m
    return m


def _mat(batch, n, layout, dtype, seed, dev="cuda"):
    if layout == "S":
        t = G.spd_packed(batch, n, dtype, seed=seed)
    else:
        t = 1 + torch.rand(batch, 1 if layout == "E" else n, dtype=F64, generator=G.gen(seed)).to(dtype)
    return t.to(dev)


def _vec(batch, n, dtype, seed, dev="cuda"):
    return G.vectors(batch, n, dtype, seed=seed).to(dev)


def _leaf(t):
    return t.detach().clone().requires_grad_()


def _gradcheck(fn, *inputs):
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-7, rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["S", "D", "E"])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_matvec_family(nfm, n, layout):
    m, v, i = _leaf(_mat(3, n, layout, F64, n)), _leaf(_vec(3, n, F64, 1)), _leaf(_vec(3, n, F64, 2))
    _gradcheck(nfm.sym_matvec, m, v)
    _gradcheck(nfm.sym_addmatvec, i, m, v)
    _gradcheck(nfm.sym_submatvec, i, m, v)


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["none", "float", "sequence", "tensor1d", "voxel"])
@pytest.mark.parametrize("method", ["auto", "ldl", "lu"])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_solve(nfm, n, method, reg):
    m, v = _leaf(_mat(3, n, "S", F64, n)), _leaf(_vec(3, n, F64, 1))
    if reg in ("none", "float", "sequence"):
        d = {"none": None, "float": 0.5, "sequence": [0.1, 0.2][:n]}[reg]
        _gradcheck(lambda m, v: nfm.sym_solve(m, v, d, method=method), m, v)
    else:
        d = _leaf(torch.rand(n if reg == "tensor1d" else (3, n), dtype=F64, generator=G.gen(5)).cuda())
        _gradcheck(lambda m, v, d: nfm.sym_solve(m, v, d, method=method), m, v, d)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["D", "E"])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_solve_diagonal_layouts(nfm, n, layout):
    m, v = _leaf(_mat(3, n, layout, F64, n)), _leaf(_vec(3, n, F64, 1))
    d = _leaf(torch.rand(3, n, dtype=F64, generator=G.gen(5)).cuda())
    _gradcheck(lambda m, v, d: nfm.sym_solve(m, v, d), m, v, d)
    _gradcheck(lambda m, v: nfm.sym_solve(m, v, eps=0.25), m, v)


@pytest.mark.gpu
@pytest.mark.parametrize("diag", [False, True])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_invert_and_det(nfm, n, diag):
    m = _leaf(_mat(3, n, "S", F64, n))
    _gradcheck(lambda m: nfm.sym_invert(m, diag), m)
    if not diag:
        _gradcheck(nfm.sym_det, _leaf(m / n))


BIG = 65536 + 37          # full TMA tiles, a partial tile and a strided tail


def _bars(dtype):
    return TOL[dtype]


_REF = {}


def _reference(kind, n, dtype):
    """Inputs in `dtype`, and the gradients of autograd through the oracle on those inputs in fp64."""
    key = (kind, n, dtype)
    if key not in _REF:
        nn = n * (n + 1) // 2
        p = G.spd_packed(BIG, n, dtype, seed=100 + n)
        v, g = G.vectors(BIG, n, dtype, seed=7), G.vectors(BIG, n, dtype, seed=8)
        if kind == "matvec":
            ins, fn = [p, v], lambda p, v: P.sym_submatvec(torch.zeros_like(v), p, v)
        elif kind == "solve":
            d = torch.rand(BIG, n, generator=G.gen(9), dtype=F64).to(dtype)
            ins, fn = [p, v, d], lambda p, v, d: P.sym_solve(p, v, d)
        elif kind == "invert":
            g = G.vectors(BIG, nn, dtype, seed=8)
            ins, fn = [p], lambda p: P.sym_invert(p)
        elif kind == "invert_diag":
            ins, fn = [p], lambda p: P.sym_invert(p, True)
        else:
            p = (p.to(F64) / n).to(dtype)
            g = G.vectors(BIG, 1, dtype, seed=8)[:, 0]
            ins, fn = [p], lambda p: torch.det(P.sym_to_full(p))
        grads = _oracle_grads(fn, [t.to(F64) for t in ins], g.to(F64))
        _REF[key] = (ins, g, grads)
    return _REF[key]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["matvec", "solve", "invert", "invert_diag", "det"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", NS)
def test_gradient_parity_at_the_bars(nfm, n, dtype, kind):
    ins, g, ref = _reference(kind, n, dtype)
    leaves = [_leaf(t.cuda()) for t in ins]
    fn = {"matvec": lambda p, v: nfm.sym_submatvec(torch.zeros_like(v), p, v),
          "solve": lambda p, v, d: nfm.sym_solve(p, v, d), "invert": lambda p: nfm.sym_invert(p),
          "invert_diag": lambda p: nfm.sym_invert(p, True), "det": nfm.sym_det}[kind]
    got = torch.autograd.grad(fn(*leaves), leaves, g.cuda())
    for a, b in zip(got, ref):
        assert a.dtype == dtype
        assert G.rel_err(a, b) < _bars(dtype), (kind, n, dtype, G.rel_err(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [3, 6, 10])
def test_new_kernels_take_the_tma_path_on_dense_fields(nfm, n, dtype):
    from nitorch_fastmath_b200 import _autograd as A
    lib = _lib.load()
    nn = n * (n + 1) // 2
    u, w = _vec(8192, n, dtype, 1), _vec(8192, n, dtype, 2)
    for layout in LAYOUTS.values():
        A.outer2(u, w, layout, -1)
        assert lib.nfm_last_path_was_tma() == 1
    b = _mat(8192, n, "S", dtype, 3)
    A.invert_backward(b, _vec(8192, nn, dtype, 4), False)
    assert lib.nfm_last_path_was_tma() == 1
    A.invert_backward(b, u, True)
    assert lib.nfm_last_path_was_tma() == 1
    A.det_backward(b, u[:, 0].contiguous())
    assert lib.nfm_last_path_was_tma() == 1
    torch.cuda.synchronize()
    # the kernels' values against the formulas (the strided tail is in the parity test)
    ud, wd, bd = u.double().cpu(), w.double().cpu(), b.double().cpu()
    eps = torch.finfo(dtype).eps
    for name, layout in LAYOUTS.items():
        got, ref = A.outer2(u, w, layout, 1).double().cpu(), ref_S(ud, wd, name)
        if name == "E":   # a dot product: the error bound is relative to sum |u_i w_i|, not to the (cancelling) sum
            assert ((got - ref).abs() <= 2 * n * eps * ref_S(ud.abs(), wd.abs(), "E")).all()
        else:
            assert G.rel_err(got, ref) < TOL[dtype]
    gd = u[:, 0].double().cpu()
    assert G.rel_err(A.det_backward(b, u[:, 0].contiguous()), ref_det(bd, gd)) < TOL[dtype] * 10 * n


def _grads(fn, inputs, g):
    leaves = [_leaf(t) for t in inputs]
    return torch.autograd.grad(fn(*leaves), leaves, g)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 4])
def test_det_gradient_is_finite_for_singular_matrices(nfm, n):
    """Orders up to 4 use the closed-form adjugate: det A = 0 still has the gradient adj(A)."""
    m = _leaf(nfm.sym_outer(_vec(8, n, F64, 1)))     # rank 1
    g, = torch.autograd.grad(nfm.sym_det(m).sum(), m)
    assert torch.isfinite(g).all()
    ref = ref_det_adjugate(m.detach().cpu())
    assert (g.cpu() - ref).abs().max() <= 1e-12 * max(1.0, ref.abs().max().item())


def ref_det_adjugate(p):
    """Gradient of det at any p through the cofactors of the expanded matrix."""
    a = P.sym_to_full(p)
    n = a.shape[-1]
    cof = torch.empty_like(a)
    for i in range(n):
        for j in range(n):
            keep_r = [r for r in range(n) if r != i]
            keep_c = [c for c in range(n) if c != j]
            cof[..., i, j] = (-1) ** (i + j) * torch.det(a[..., keep_r, :][..., :, keep_c])
    return _pack_sym_grad(cof)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 6])
def test_broadcast_gradients_are_sums_of_per_matrix_gradients(nfm, n):
    nn, B, X = n * (n + 1) // 2, 4, 5
    shared = _mat(1, n, "S", F64, 1)[0]
    v, g = _vec(B, n, F64, 2), _vec(B, n, F64, 3)
    cases = [(lambda m, v: nfm.sym_matvec(m, v)), (lambda m, v: nfm.sym_solve(m, v)),
             (lambda m, v: nfm.sym_submatvec(v, m, v))]
    for fn in cases:
        gm, gv = _grads(fn, [shared, v], g)
        em, ev = _grads(fn, [shared.expand(B, nn).contiguous(), v], g)
        assert gm.shape == shared.shape and _close(gm, em.sum(0)) and _close(gv, ev)
    # partially broadcast: one field (1, X, NN) for a batch of vector fields (B, X, N)
    field = _mat(X, n, "S", F64, 4).view(1, X, nn)
    vb, gb = _vec(B * X, n, F64, 5).view(B, X, n), _vec(B * X, n, F64, 6).view(B, X, n)
    d = torch.rand(X, n, dtype=F64, generator=G.gen(7)).cuda()
    for fn in cases + [lambda m, v: nfm.sym_solve(m, v, d)]:
        gm, gv = _grads(fn, [field, vb], gb)
        em, ev = _grads(fn, [field.expand(B, X, nn).contiguous(), vb], gb)
        assert gm.shape == field.shape and _close(gm, em.sum(0, keepdim=True)) and _close(gv, ev)
    # a 1-D regulariser that requires grad collects the gradient of every matrix
    dl = _leaf(torch.rand(n, dtype=F64, generator=G.gen(8)).cuda())
    m = _mat(B, n, "S", F64, 9)
    gd, = torch.autograd.grad(nfm.sym_solve(m, v, dl), dl, g)
    dv = _leaf(dl.detach().expand(B, n).contiguous())
    ed, = torch.autograd.grad(nfm.sym_solve(m, v, dv), dv, g)
    assert _close(gd, ed.sum(0))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6])
def test_strided_and_offset_views_give_the_gradients_of_contiguous_copies(nfm, n):
    nn, B = n * (n + 1) // 2, 300
    m, v, g = _mat(B, n, "S", F64, 1), _vec(B, n, F64, 2), _vec(B, n, F64, 3)
    m_cf = m.t().contiguous().t()                         # coefficient-first storage viewed coefficient-last
    v_cf = v.t().contiguous().t()
    m_off = torch.cat([m.new_zeros(nn + 1), m.flatten()])[nn + 1:].view(B, nn)[1:]   # storage offset
    v_off = torch.cat([v.new_zeros(1), v.flatten()])[1:].view(B, n)[1:]
    for fn in [lambda m, v: nfm.sym_solve(m, v), lambda m, v: nfm.sym_addmatvec(v, m, v),
               lambda m, v: nfm.sym_invert(m)[..., :n] * v, lambda m, v: nfm.sym_det(m)[..., None] * v]:
        ref = _grads(fn, [m, v], g)
        for mm, vv in [(m_cf, v_cf)]:
            got = _grads(fn, [mm, vv], g)
            assert all(_close(a, b) for a, b in zip(got, ref))
        got = _grads(fn, [m_off, v_off], g[1:])
        ref1 = _grads(fn, [m[1:].contiguous(), v[1:].contiguous()], g[1:])
        assert all(_close(a, b) for a, b in zip(got, ref1))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 5])
def test_inplace_variants_on_non_leaf_inputs(nfm, n):
    m0, v0, i0 = _mat(16, n, "S", F64, 1), _vec(16, n, F64, 2), _vec(16, n, F64, 3)
    g = _vec(16, n, F64, 4)
    nn = n * (n + 1) // 2
    gn = _vec(16, nn, F64, 5)

    def via(fn_inplace, fn, inputs, which, grad):
        leaves = [_leaf(t) for t in inputs]
        work = [t * 1 for t in leaves]
        out = fn_inplace(*work)
        assert out is work[which]
        a = torch.autograd.grad(out, leaves, grad)
        leaves = [_leaf(t) for t in inputs]
        b = torch.autograd.grad(fn(*leaves), leaves, grad)
        assert all(_close(x, y) for x, y in zip(a, b))

    via(lambda m, v: nfm.sym_solve_(m, v), lambda m, v: nfm.sym_solve(m, v), [m0, v0], 1, g)
    via(lambda m, v: nfm.sym_solve_(m, v, 0.5), lambda m, v: nfm.sym_solve(m, v, 0.5), [m0, v0], 1, g)
    via(lambda m: nfm.sym_invert_(m), lambda m: nfm.sym_invert(m), [m0], 0, gn)
    via(lambda i, m, v: nfm.sym_addmatvec_(i, m, v), lambda i, m, v: nfm.sym_addmatvec(i, m, v), [i0, m0, v0], 0, g)
    via(lambda i, m, v: nfm.sym_submatvec_(i, m, v), lambda i, m, v: nfm.sym_submatvec(i, m, v), [i0, m0, v0], 0, g)
    with pytest.raises(RuntimeError):           # torch's own error for a leaf that requires grad
        nfm.sym_solve_(m0, _leaf(v0))


@pytest.mark.gpu
def test_error_paths(nfm):
    m, v = _leaf(_mat(4, 3, "S", F64, 1)), _leaf(_vec(4, 3, F64, 2))
    with pytest.raises(RuntimeError):
        nfm.sym_solve(m, v, out=torch.empty(4, 3, dtype=F64, device="cuda"))
    with pytest.raises(RuntimeError):
        nfm.sym_matvec(m, v, out=torch.empty(4, 3, dtype=F64, device="cuda"))
    with pytest.raises(RuntimeError):
        nfm.sym_invert(m, out=torch.empty(4, 6, dtype=F64, device="cuda"))
    full = _leaf(torch.eye(3, dtype=F64, device="cuda").flatten().expand(4, 9) * 2)
    with pytest.raises(NotImplementedError):
        nfm.sym_solve(full, v)
    with pytest.raises(NotImplementedError):
        nfm.sym_matvec(full, v)
    for fn in [lambda: nfm.sym_solve(m, v), lambda: nfm.sym_matvec(m, v), lambda: nfm.sym_invert(m)[..., :3] * v,
               lambda: nfm.sym_det(m)]:
        gm, = torch.autograd.grad(fn().sum(), m, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(gm.sum(), m)


@pytest.mark.gpu
def test_backward_follows_a_side_stream_forward(nfm):
    n = 6
    m, v, g = _mat(200000, n, "S", torch.float32, 1), _vec(200000, n, torch.float32, 2), _vec(200000, n, torch.float32, 3)
    ref = _grads(lambda m, v: nfm.sym_solve(m, v), [m, v], g)
    ml, vl = _leaf(m), _leaf(v)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        x = nfm.sym_solve(ml, vl)
        loss = (x * g).sum()
    torch.cuda.current_stream().wait_stream(side)
    got = torch.autograd.grad(loss, (ml, vl))
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(got, ref))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 7])
def test_cpu_operands_get_the_gradients_of_cuda_operands(nfm, n):
    m, v, g = _mat(64, n, "S", F64, 1, "cpu"), _vec(64, n, F64, 2, "cpu"), _vec(64, n, F64, 3, "cpu")
    d = torch.rand(64, n, dtype=F64, generator=G.gen(4))
    gi = _vec(64, n * (n + 1) // 2, F64, 5, "cpu")
    cases = [(lambda m, v, d: nfm.sym_solve(m, v, d), [m, v, d], g), (lambda m, v: nfm.sym_submatvec(v, m, v), [m, v], g),
             (lambda m: nfm.sym_invert(m), [m], gi), (lambda m: nfm.sym_invert(m, True), [m], g),
             (lambda m: nfm.sym_det(m), [m], g[:, 0])]
    for fn, ins, gg in cases:
        got = _grads(fn, ins, gg)
        ref = _grads(fn, [t.cuda() for t in ins], gg.cuda())
        assert all(a.device.type == "cpu" and _close(a, b) for a, b in zip(got, ref))


@pytest.mark.gpu
def test_mixed_and_half_dtypes_return_gradients_in_the_input_dtypes(nfm):
    m, v = _leaf(_mat(32, 3, "S", F64, 1)), _leaf(_vec(32, 3, torch.float32, 2))
    gm, gv = torch.autograd.grad(nfm.sym_solve(m, v).sum(), (m, v))
    assert gm.dtype == F64 and gv.dtype == torch.float32
    mh, vh = _leaf(_mat(32, 3, "S", torch.half, 1)), _leaf(_vec(32, 3, torch.half, 2))
    gm, gv = torch.autograd.grad(nfm.sym_matvec(mh, vh).float().sum(), (mh, vh))
    assert gm.dtype == torch.half and gv.dtype == torch.half
    ref = _grads(lambda m, v: nfm.sym_matvec(m, v), [mh.detach().float(), vh.detach().float()],
                 torch.ones(32, 3, device="cuda"))
    assert _close(gm.float(), ref[0], 1e-3) and _close(gv.float(), ref[1], 1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6])
def test_no_grad_behaviour_is_unchanged(nfm, n):
    m, v, i = _mat(4096, n, "S", torch.float32, 1), _vec(4096, n, torch.float32, 2), _vec(4096, n, torch.float32, 3)
    calls = [lambda m, v, i: nfm.sym_matvec(m, v), lambda m, v, i: nfm.sym_addmatvec(i, m, v),
             lambda m, v, i: nfm.sym_submatvec(i, m, v), lambda m, v, i: nfm.sym_solve(m, v, 0.1),
             lambda m, v, i: nfm.sym_invert(m), lambda m, v, i: nfm.sym_invert(m, True), lambda m, v, i: nfm.sym_det(m)]
    for call in calls:
        b0 = _lib.launch_count()
        plain = call(m, v, i)
        d_plain = _lib.launch_count() - b0
        ml, vl, il = _leaf(m), _leaf(v), _leaf(i)
        with torch.no_grad():
            b0 = _lib.launch_count()
            gated = call(ml, vl, il)
            d_gated = _lib.launch_count() - b0
        assert not plain.requires_grad and not gated.requires_grad
        assert torch.equal(plain, gated) and d_plain == d_gated
