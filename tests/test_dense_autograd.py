"""Gradients of batchdet, batchinv, batchmatvec, lmdiv and rmdiv (and through them inv,
solvevec and matvec): nitorch_fastmath_b200/_autograd.py, csrc/nfm_dense_grad.cu.

The formulas are written once here (``ref_*``) and pinned to autograd through torch /
the oracle on CPU fp64; the GPU tests run ``torch.autograd.gradcheck`` and compare the
library against those oracle gradients."""
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
KS = [1, 2, 3, 4, 5, 8]
ROWS = [1, 2, 4, 5]


# ---------------------------------------------------------------------------
# reference formulas (DESIGN.md, "Gradients")
# ---------------------------------------------------------------------------

def _symm(m):
    return 0.5 * (m + m.transpose(-1, -2))


def ref_det(a, g):
    """g adj(A)^T through the cofactors: finite for singular matrices."""
    n = a.shape[-1]
    cof = torch.empty_like(a)
    for i in range(n):
        for j in range(n):
            keep_r = [r for r in range(n) if r != i]
            keep_c = [c for c in range(n) if c != j]
            minor = a[..., keep_r, :][..., :, keep_c]
            cof[..., i, j] = (-1) ** (i + j) * (torch.det(minor) if n > 1 else torch.ones_like(a[..., 0, 0]))
    return g[..., None, None] * cof


def ref_inv(a, g, chol):
    y = P.inv(a, "chol") if chol else torch.linalg.inv(a)
    if chol:
        return -y @ _symm(g) @ y
    yt = y.transpose(-1, -2)
    return -yt @ g @ yt


def ref_lmdiv(a, b, g, chol):
    """dA, dB of X = A^-1 B."""
    x = P.lmdiv(a, b, "chol" if chol else "lu")
    u = P.lmdiv(a, g, "chol") if chol else torch.linalg.solve(a.transpose(-1, -2), g)
    da = -u @ x.transpose(-1, -2)
    return (_symm(da) if chol else da), u


def ref_rmdiv(a, b, g, chol):
    """d_a, d_b of Y = a b^-1 (a: k x n)."""
    y = _rm(a, b, chol)
    u = (P.lmdiv(b, g.transpose(-1, -2), "chol").transpose(-1, -2) if chol
         else torch.linalg.solve(b, g.transpose(-1, -2)).transpose(-1, -2))
    db = -y.transpose(-1, -2) @ u
    return u, (_symm(db) if chol else db)


def ref_matvec(a, v, g):
    return g.unsqueeze(-1) * v.unsqueeze(-2), (a.transpose(-1, -2) @ g.unsqueeze(-1)).squeeze(-1)


def _rm(a, b, chol):
    """a b^-1 through torch: solve with b^T (lu) or the Cholesky factor of b's lower triangle."""
    return P.lmdiv(b, a.transpose(-1, -2), "chol").transpose(-1, -2) if chol else \
        torch.linalg.solve(b.transpose(-1, -2), a.transpose(-1, -2)).transpose(-1, -2)


def _oracle_grads(fn, inputs, g):
    inputs = [t.detach().clone().requires_grad_() for t in inputs]
    return torch.autograd.grad(fn(*inputs), inputs, g)


def _close(a, b, tol=1e-10):
    return G.rel_err(a, b, 2 if a.dim() >= 2 and b.dim() >= 2 else 1) < tol


# ---------------------------------------------------------------------------
# CPU: the formulas against autograd in fp64
# ---------------------------------------------------------------------------

@pytest.mark.parametrize("n", NS)
def test_det_formula(n):
    a = G.dense_shifted(5, n, F64, seed=n) / 10
    g = torch.randn(5, dtype=F64, generator=G.gen(3))
    fn = P.closed_det if n <= 3 else torch.det
    ga, = _oracle_grads(fn, [a], g)
    assert _close(ga, ref_det(a, g))


@pytest.mark.parametrize("chol", [False, True])
@pytest.mark.parametrize("n", NS)
def test_inv_formula(n, chol):
    a = G.dense_spd(5, n, F64, seed=n) if chol else G.dense_shifted(5, n, F64, seed=n)
    g = G.vectors((5, n), n, F64, seed=3)
    ga, = _oracle_grads(lambda a: P.inv(a, "chol" if chol else "lu"), [a], g)
    assert _close(ga, ref_inv(a, g, chol))
    if 2 <= n <= 3 and not chol:     # the closed forms with their determinant shift
        gc, = _oracle_grads(P.closed_inv, [a], g)
        assert _close(gc, ref_inv(a, g, False))


@pytest.mark.parametrize("chol", [False, True])
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("n", NS)
def test_lmdiv_formula(n, k, chol):
    a = G.dense_spd(4, n, F64, seed=n) if chol else G.dense_shifted(4, n, F64, seed=n)
    b, g = G.vectors((4, n), k, F64, seed=1), G.vectors((4, n), k, F64, seed=2)
    ga, gb = _oracle_grads(lambda a, b: P.lmdiv(a, b, "chol" if chol else "lu"), [a, b], g)
    da, db = ref_lmdiv(a, b, g, chol)
    assert _close(ga, da) and _close(gb, db)


@pytest.mark.parametrize("chol", [False, True])
@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("n", NS)
def test_rmdiv_formula(n, rows, chol):
    b = G.dense_spd(4, n, F64, seed=n) if chol else G.dense_shifted(4, n, F64, seed=n)
    a, g = G.vectors((4, rows), n, F64, seed=1), G.vectors((4, rows), n, F64, seed=2)
    ga, gb = _oracle_grads(lambda a, b: _rm(a, b, chol), [a, b], g)
    da, db = ref_rmdiv(a, b, g, chol)
    assert _close(ga, da) and _close(gb, db)


@pytest.mark.parametrize("m,n", [(1, 1), (3, 3), (10, 10), (3, 5), (5, 3), (1, 7), (12, 4)])
def test_matvec_formula(m, n):
    a, v, g = G.vectors((4, m), n, F64, seed=1), G.vectors(4, n, F64, seed=2), G.vectors(4, m, F64, seed=3)
    ga, gv = _oracle_grads(P.batchmatvec, [a, v], g)
    da, dv = ref_matvec(a, v, g)
    assert _close(ga, da) and _close(gv, dv)


def test_backward_entry_points_reject_bad_arguments_without_a_gpu():
    lib = _lib.load()
    buf = ctypes.create_string_buffer(4096)
    q = ctypes.addressof(buf)
    F32, LU, LDL = _lib.F32, _lib.ALGO_LU, _lib.ALGO_LDL
    # nfm_batch_det_backward(dtype, n, batch, mat, ms, grad, gs, out, os, stream)
    assert lib.nfm_batch_det_backward(F32, 11, 4, q, 121, q, 1, q, 121, None) == -1
    assert lib.nfm_batch_det_backward(F32, 0, 4, q, 1, q, 1, q, 1, None) == -1
    assert lib.nfm_batch_det_backward(7, 3, 4, q, 9, q, 1, q, 9, None) == -1
    assert lib.nfm_batch_det_backward(F32, 3, 4, None, 9, q, 1, q, 9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, 4, q, 9, None, 1, q, 9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, 4, q, 9, q, 1, None, 9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, 4, q, -9, q, 1, q, 9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, 4, q, 9, q, 1, q, -9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, -4, q, 9, q, 1, q, 9, None) == -2
    assert lib.nfm_batch_det_backward(F32, 3, 0, q, 9, q, 1, q, 9, None) == 0
    # nfm_batch_inv_backward(dtype, n, sym, batch, inv, is, grad, gs, out, os, stream)
    assert lib.nfm_batch_inv_backward(F32, 11, 0, 4, q, 121, q, 121, q, 121, None) == -1
    assert lib.nfm_batch_inv_backward(7, 3, 0, 4, q, 9, q, 9, q, 9, None) == -1
    assert lib.nfm_batch_inv_backward(F32, 3, 2, 4, q, 9, q, 9, q, 9, None) == -1
    assert lib.nfm_batch_inv_backward(F32, 3, 0, 4, None, 9, q, 9, q, 9, None) == -2
    assert lib.nfm_batch_inv_backward(F32, 3, 1, 4, q, 9, None, 9, q, 9, None) == -2
    assert lib.nfm_batch_inv_backward(F32, 3, 0, 4, q, 9, q, 9, None, 9, None) == -2
    assert lib.nfm_batch_inv_backward(F32, 3, 0, 4, q, 9, q, -9, q, 9, None) == -2
    assert lib.nfm_batch_inv_backward(F32, 3, 0, -4, q, 9, q, 9, q, 9, None) == -2
    assert lib.nfm_batch_inv_backward(F32, 3, 1, 0, q, 9, q, 9, q, 9, None) == 0
    # nfm_batch_outer(dtype, m, n, k, order, sym, sign, batch, u, us, w, ws, out, os, stream)
    assert lib.nfm_batch_outer(7, 3, 3, 2, 0, 0, 1, 4, q, 6, q, 6, q, 9, None) == -1
    assert lib.nfm_batch_outer(F32, 3, 3, 2, 2, 0, 1, 4, q, 6, q, 6, q, 9, None) == -1
    assert lib.nfm_batch_outer(F32, 3, 3, 2, 0, 2, 1, 4, q, 6, q, 6, q, 9, None) == -1
    assert lib.nfm_batch_outer(F32, 3, 4, 2, 0, 1, 1, 4, q, 6, q, 8, q, 12, None) == -1   # sym needs m == n
    assert lib.nfm_batch_outer(F32, 0, 3, 2, 0, 0, 1, 4, q, 6, q, 6, q, 9, None) == -2
    assert lib.nfm_batch_outer(F32, 3, 3, 0, 0, 0, 1, 4, q, 6, q, 6, q, 9, None) == -2
    assert lib.nfm_batch_outer(F32, 3, 3, 2, 0, 0, 0, 4, q, 6, q, 6, q, 9, None) == -2
    assert b"sign" in lib.nfm_last_error_string()
    for m, n, k in [(3, 3, 2), (3, 5, 1), (4, 4, 6)]:       # register kernels and the run-time-sized kernel
        us, ws, os_ = m * k, n * k, m * n
        assert lib.nfm_batch_outer(F32, m, n, k, 0, 0, 1, 4, None, us, q, ws, q, os_, None) == -2
        assert lib.nfm_batch_outer(F32, m, n, k, 0, 0, 1, 4, q, us, None, ws, q, os_, None) == -2
        assert lib.nfm_batch_outer(F32, m, n, k, 0, 0, 1, 4, q, us, q, ws, None, os_, None) == -2
        assert lib.nfm_batch_outer(F32, m, n, k, 0, 0, 1, 4, q, -us, q, ws, q, os_, None) == -2
        assert lib.nfm_batch_outer(F32, m, n, k, 1, 0, -1, -4, q, us, q, ws, q, os_, None) == -2
        assert lib.nfm_batch_outer(F32, m, n, k, 0, 0, 1, 0, q, us, q, ws, q, os_, None) == 0
    # nfm_batch_tsolve(dtype, n, k, right, algo, batch, mat, as, b, bs, out, os, stream)
    assert lib.nfm_batch_tsolve(F32, 11, 2, 0, LU, 4, q, 121, q, 22, q, 22, None) == -1
    assert lib.nfm_batch_tsolve(7, 3, 2, 0, LU, 4, q, 9, q, 6, q, 6, None) == -1
    assert lib.nfm_batch_tsolve(F32, 3, 2, 2, LU, 4, q, 9, q, 6, q, 6, None) == -1
    assert lib.nfm_batch_tsolve(F32, 3, 2, 0, _lib.ALGO_WARP, 4, q, 9, q, 6, q, 6, None) == -1
    assert lib.nfm_batch_tsolve(F32, 3, 0, 0, LU, 4, q, 9, q, 6, q, 6, None) == -2
    for k in (1, 3, 8):
        for right, algo in [(0, LU), (1, LDL)]:
            bl = 3 * k
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, 4, None, 9, q, bl, q, bl, None) == -2
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, 4, q, 9, None, bl, q, bl, None) == -2
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, 4, q, 9, q, bl, None, bl, None) == -2
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, 4, q, 9, q, -bl, q, bl, None) == -2
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, -4, q, 9, q, bl, q, bl, None) == -2
            assert lib.nfm_batch_tsolve(F32, 3, k, right, algo, 0, q, 9, q, bl, q, bl, None) == 0
    # nfm_batch_tmatvec(dtype, m, n, batch, mat, ms, vec, vs, out, os, stream)
    assert lib.nfm_batch_tmatvec(7, 3, 3, 4, q, 9, q, 3, q, 3, None) == -1
    for m, n in [(3, 3), (3, 5)]:
        assert lib.nfm_batch_tmatvec(F32, 0, n, 4, q, 0, q, 0, q, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, 4, None, m * n, q, m, q, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, 4, q, m * n, None, m, q, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, 4, q, m * n, q, m, None, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, 4, q, m * n, q, -m, q, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, -4, q, m * n, q, m, q, n, None) == -2
        assert lib.nfm_batch_tmatvec(F32, m, n, 0, q, m * n, q, m, q, n, None) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_gradient_path_fails_loudly_without_cuda():
    import nitorch_fastmath_b200 as nfm
    a = (torch.rand(8, 3, 3) + 3 * torch.eye(3)).requires_grad_()
    v = torch.rand(8, 3).requires_grad_()
    calls = [lambda: nfm.batchdet(a), lambda: nfm.batchinv(a), lambda: nfm.batchmatvec(a, v),
             lambda: nfm.lmdiv(a, v[..., None]), lambda: nfm.rmdiv(v[..., None, :], a), lambda: nfm.inv(a),
             lambda: nfm.solvevec(a, v), lambda: nfm.matvec(a, v)]
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


def _leaf(t):
    return t.detach().clone().requires_grad_()


def _gradcheck(fn, *inputs):
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-7, rtol=1e-5)


def _a(batch, n, dtype, seed, chol=False, dev="cuda"):
    return (G.dense_spd(batch, n, dtype, seed=seed) if chol else G.dense_shifted(batch, n, dtype, seed=seed)).to(dev)


def _v(batch, n, dtype, seed, dev="cuda"):
    return G.vectors(batch, n, dtype, seed=seed).to(dev)


def _grads(fn, inputs, g):
    leaves = [_leaf(t) for t in inputs]
    return torch.autograd.grad(fn(*leaves), leaves, g)


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
def test_gradcheck_det_inv_and_matvec(nfm, n):
    a = _leaf(_a(2, n, F64, n) / 4)
    _gradcheck(nfm.batchdet, a)
    for method, reg in [("auto", True), ("auto", False), ("lu", True)]:
        _gradcheck(lambda a: nfm.batchinv(a, method=method, regularise=reg), a)
    _gradcheck(lambda a: nfm.inv(a), a)
    s = _leaf(_a(2, n, F64, n, chol=True))
    _gradcheck(lambda s: nfm.batchinv(_symm(s), method="chol"), s)
    _gradcheck(lambda s: nfm.inv(_symm(s), method="chol"), s)
    for m in {n, n + 2, max(1, n - 3)}:
        _gradcheck(nfm.batchmatvec, _leaf(_v((2, m), n, F64, 1)), _leaf(_v(2, n, F64, 2)))
    _gradcheck(nfm.matvec, a, _leaf(_v(2, n, F64, 2)))


@pytest.mark.gpu
@pytest.mark.parametrize("chol", [False, True])
@pytest.mark.parametrize("n", NS)
def test_gradcheck_lmdiv_rmdiv(nfm, n, chol):
    method = "chol" if chol else "lu"
    a = _leaf(_a(2, n, F64, n, chol))
    prep = _symm if chol else (lambda t: t)
    for k in KS:
        _gradcheck(lambda a, b: nfm.lmdiv(prep(a), b, method=method), a, _leaf(_v((2, n), k, F64, k)))
    for rows in ROWS:
        _gradcheck(lambda x, a: nfm.rmdiv(x, prep(a), method=method), _leaf(_v((2, rows), n, F64, rows)), a)
    _gradcheck(lambda a, v: nfm.solvevec(prep(a), v, method=method), a, _leaf(_v(2, n, F64, 3)))


BIG = 65536 + 37          # full TMA tiles, a partial tile and a strided tail; ragged
_REF = {}


def _case(kind, n, dtype, k):
    """Inputs in `dtype` and the fp64 oracle gradients on those inputs."""
    key = (kind, n, dtype, k)
    if key not in _REF:
        chol = kind.endswith("chol")
        a = (G.dense_spd if chol else G.dense_shifted)(BIG, n, dtype, seed=100 + n)
        if kind == "det":
            a = (a.to(F64) / 10).to(dtype)
            ins, g, fn = [a], G.vectors(BIG, 1, dtype, seed=8)[:, 0], torch.det
        elif kind.startswith("inv"):
            ins, g, fn = [a], G.vectors((BIG, n), n, dtype, seed=8), lambda a: P.inv(a, "chol" if chol else "lu")
        elif kind.startswith("lmdiv"):
            ins = [a, G.vectors((BIG, n), k, dtype, seed=7)]
            g, fn = G.vectors((BIG, n), k, dtype, seed=8), lambda a, b: P.lmdiv(a, b, "chol" if chol else "lu")
        elif kind.startswith("rmdiv"):
            ins = [G.vectors((BIG, k), n, dtype, seed=7), a]
            g, fn = G.vectors((BIG, k), n, dtype, seed=8), lambda x, a: _rm(x, a, chol)
        else:
            ins, g, fn = [a, G.vectors(BIG, n, dtype, seed=7)], G.vectors(BIG, n, dtype, seed=8), P.batchmatvec
        _REF[key] = (ins, g, _oracle_grads(fn, [t.to(F64) for t in ins], g.to(F64)))
    return _REF[key]


PARITY = ([("det", 0), ("inv", 0), ("inv_chol", 0), ("matvec", 0)]
          + [(f"lmdiv{c}", k) for c in ("", "_chol") for k in (1, 3, 8)] + [(f"rmdiv{c}", r) for c in ("", "_chol") for r in (1, 3)])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,k", PARITY)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [2, 3, 4, 7, 10])
def test_gradient_parity_at_the_bars(nfm, n, dtype, kind, k):
    ins, g, ref = _case(kind, n, dtype, k)
    leaves = [_leaf(t.cuda()) for t in ins]
    fn = {"det": nfm.batchdet, "inv": nfm.batchinv, "inv_chol": lambda a: nfm.batchinv(a, method="chol"),
          "matvec": nfm.batchmatvec, "lmdiv": nfm.lmdiv, "lmdiv_chol": lambda a, b: nfm.lmdiv(a, b, method="chol"),
          "rmdiv": nfm.rmdiv, "rmdiv_chol": lambda x, a: nfm.rmdiv(x, a, method="chol")}[kind]
    got = torch.autograd.grad(fn(*leaves), leaves, g.cuda())
    for a, b in zip(got, ref):
        assert a.dtype == dtype
        assert G.rel_err(a, b, 2 if b.dim() == 3 else 1) < TOL[dtype], (kind, n, dtype, k, G.rel_err(a, b, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [3, 4, 6, 10])
def test_new_kernels_take_the_tma_path_on_dense_aligned_fields(nfm, n, dtype):
    """The light backward kernels run on the TMA tile kernel (path 1); the pivoted ones (the
    determinant backward from n = 4, the transposed LU solves) on the tile or warp-pool kernel
    (1 / 3) as their forward kernels do, and the transposed single-column solve on the staged
    many-right-hand-side kernel (4)."""
    from nitorch_fastmath_b200 import _autograd as A
    lib = _lib.load()
    B = 8192
    a, y = _a(B, n, dtype, 1), _a(B, n, dtype, 2)
    gm = _v((B, n), n, dtype, 3)
    # fp64 n = 9, 10: two 81 / 100-double inputs and the output do not fit a shared-memory ring of the
    # smallest tile (DESIGN.md section 6): the strided kernel (path 0)
    inv_path = 0 if dtype == F64 and n >= 9 else 1
    A.dense_inv_backward(y, gm, False)
    assert lib.nfm_last_path_was_tma() == inv_path
    A.dense_inv_backward(y, gm, True)
    assert lib.nfm_last_path_was_tma() == inv_path
    for k in (1, 2, 4):
        u, w = _v((B, n), k, dtype, 4), _v((B, n), k, dtype, 5)
        for rows in (False, True):
            for sym in (False, True):
                if rows:    # the same records read as k x n
                    A.dense_outer(u.view(B, k, n), w.view(B, k, n), rows, sym, -1)
                else:
                    A.dense_outer(u, w, rows, sym, -1)
                assert lib.nfm_last_path_was_tma() == 1
        A.dense_tsolve(a, u, False, _lib.ALGO_LU)
        assert lib.nfm_last_path_was_tma() in ((4,) if k == 1 else (1, 3))
    A.dense_tmatvec(a, _v(B, n, dtype, 6))
    assert lib.nfm_last_path_was_tma() == 1
    A.dense_det_backward(a, _v(B, 1, dtype, 7)[:, 0].contiguous())
    assert lib.nfm_last_path_was_tma() in ((1,) if n <= 3 else (1, 3))
    torch.cuda.synchronize()
    # the values of every kernel on these launches against the formulas
    ad, yd, gd = a.double().cpu(), y.double().cpu(), gm.double().cpu()
    yt = yd.transpose(-1, -2)
    assert G.rel_err(A.dense_inv_backward(y, gm, False), -yt @ gd @ yt, 2) < TOL[dtype] * 10
    assert G.rel_err(A.dense_inv_backward(y, gm, True), -yd @ _symm(gd) @ yd, 2) < TOL[dtype] * 10
    u, w = _v((B, n), 3, dtype, 4), _v((B, n), 3, dtype, 5)
    ud, wd = u.double().cpu(), w.double().cpu()
    assert G.rel_err(A.dense_outer(u, w, False, True, -1), -_symm(ud @ wd.transpose(-1, -2)), 2) < TOL[dtype] * 10
    assert G.rel_err(A.dense_outer(u.transpose(-1, -2).contiguous(), w.transpose(-1, -2).contiguous(), True, False, 1),
                     ud @ wd.transpose(-1, -2), 2) < TOL[dtype] * 10
    assert G.rel_err(A.dense_tsolve(a, u, False, _lib.ALGO_LU), torch.linalg.solve(ad.transpose(-1, -2), ud), 2) < TOL[dtype] * 10
    assert G.rel_err(A.dense_tmatvec(a, u[..., 0].contiguous()),
                     (ad.transpose(-1, -2) @ ud[..., :1]).squeeze(-1)) < TOL[dtype] * 10


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3])
def test_det_gradient_of_singular_matrices_is_the_adjugate(nfm, n):
    x = _v(8, n, F64, 1)
    a = _leaf(x.unsqueeze(-1) * _v(8, n, F64, 2).unsqueeze(-2))      # rank 1
    a2 = _leaf(torch.zeros(1, n, n, dtype=F64, device="cuda"))
    for m in (a, a2):
        g, = torch.autograd.grad(nfm.batchdet(m).sum(), m)
        ref = ref_det(m.detach().cpu(), torch.ones(m.shape[0], dtype=F64))
        assert torch.isfinite(g).all()
        assert (g.cpu() - ref).abs().max() <= 1e-13 * max(1.0, ref.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 5])
def test_broadcast_gradients_are_sums_of_per_matrix_gradients(nfm, n):
    B = 6
    shared = _a(1, n, F64, 1)[0]
    bk, gk = _v((B, n), 3, F64, 2), _v((B, n), 3, F64, 3)
    rows, gr = _v((B, 2), n, F64, 4), _v((B, 2), n, F64, 5)
    v, gv = _v(B, n, F64, 6), _v(B, n, F64, 7)
    cases = [(lambda a, b: nfm.lmdiv(a, b), bk, gk), (lambda a, b: nfm.lmdiv(a, b, method="chol"), bk, gk),
             (lambda a, x: nfm.rmdiv(x, a), rows, gr), (lambda a, v: nfm.batchmatvec(a, v), v, gv),
             (lambda a, v: nfm.solvevec(a, v), v, gv)]
    spd = _a(1, n, F64, 1, chol=True)[0]
    for i, (fn, other, g) in enumerate(cases):
        a0 = spd if i == 1 else shared
        ga, go = _grads(fn, [a0, other], g)
        ea, eo = _grads(fn, [a0.expand(B, n, n).contiguous(), other], g)
        assert ga.shape == a0.shape and _close(ga, ea.sum(0), 1e-12) and _close(go, eo, 1e-12)
    # one vector for a batch of matrices
    mats = _a(B, n, F64, 8)
    gv1, = _grads(lambda v: nfm.batchmatvec(mats, v), [v[0]], gv)
    ev, = _grads(lambda v: nfm.batchmatvec(mats, v), [v[0].expand(B, n).contiguous()], gv)
    assert gv1.shape == (n,) and _close(gv1, ev.sum(0), 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6])
def test_offset_and_transposed_batch_views_give_the_gradients_of_contiguous_copies(nfm, n):
    B = 300
    a, b, v = _a(B, n, F64, 1), _v((B, n), 3, F64, 2), _v(B, n, F64, 3)
    g3, gv = _v((B, n), 3, F64, 4), _v(B, n, F64, 5)
    a_off = torch.cat([a.new_zeros(1), a.flatten()])[1:].view(B, n, n)[1:]      # storage offset
    a_tb = a.view(2, B // 2, n, n).transpose(0, 1).contiguous().transpose(0, 1)   # transposed batch dims
    cases = [(lambda a, b: nfm.lmdiv(a, b), b, g3), (lambda a, v: nfm.batchmatvec(a, v), v, gv),
             (lambda a, v: (nfm.batchinv(a) @ v[..., None])[..., 0], v, gv), (lambda a, v: nfm.batchdet(a)[..., None] * v, v, gv)]
    for fn, other, g in cases:
        got = _grads(fn, [a_off, other[1:]], g[1:])
        ref = _grads(fn, [a[1:].contiguous(), other[1:].contiguous()], g[1:])
        assert all(_close(x, y, 1e-12) for x, y in zip(got, ref))
        sh = (2, B // 2)
        got = _grads(fn, [a_tb, other.view(*sh, *other.shape[1:])], g.view(*sh, *g.shape[1:]))
        ref = _grads(fn, [a.view(*sh, n, n), other.view(*sh, *other.shape[1:])], g.view(*sh, *g.shape[1:]))
        assert all(_close(x, y, 1e-12) for x, y in zip(got, ref))


@pytest.mark.gpu
def test_empty_batches(nfm):
    for shape in [(0, 3, 3), (2, 0, 4, 4)]:
        a = _leaf(torch.zeros(shape, dtype=F64, device="cuda"))
        n = shape[-1]
        v = _leaf(torch.zeros(shape[:-1], dtype=F64, device="cuda"))
        for out in [nfm.batchdet(a).sum(), nfm.batchinv(a).sum(), nfm.batchmatvec(a, v).sum(), nfm.lmdiv(a, v[..., None]).sum(),
                    nfm.rmdiv(v[..., None, :], a).sum(), nfm.solvevec(a, v).sum()]:
            ga, gv = torch.autograd.grad(out, (a, v), allow_unused=True)
            assert ga is None or ga.shape == a.shape
            assert gv is None or gv.shape == v.shape
        assert n > 0
    # no right-hand side: no work, zero matrix gradient
    a = _leaf(_a(4, 3, F64, 1))
    ga, = torch.autograd.grad(nfm.lmdiv(a, torch.zeros(4, 3, 0, dtype=F64, device="cuda")).sum(), a, allow_unused=True)
    assert ga is None or (ga == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 7])
def test_cpu_operands_get_the_gradients_of_cuda_operands(nfm, n):
    a, b, v = _a(64, n, F64, 1, dev="cpu"), _v((64, n), 2, F64, 2, dev="cpu"), _v(64, n, F64, 3, dev="cpu")
    g2, gv, gi, gd = _v((64, n), 2, F64, 4, "cpu"), _v(64, n, F64, 5, "cpu"), _v((64, n), n, F64, 6, "cpu"), _v(64, 1, F64, 7, "cpu")[:, 0]
    r, gr = _v((64, 2), n, F64, 8, "cpu"), _v((64, 2), n, F64, 9, "cpu")
    cases = [(nfm.batchdet, [a], gd), (nfm.batchinv, [a], gi), (nfm.batchmatvec, [a, v], gv), (nfm.lmdiv, [a, b], g2),
             (lambda x, a: nfm.rmdiv(x, a), [r, a], gr), (nfm.solvevec, [a, v], gv)]
    for fn, ins, gg in cases:
        got = _grads(fn, ins, gg)
        ref = _grads(fn, [t.cuda() for t in ins], gg.cuda())
        assert all(x.device.type == "cpu" and _close(x, y, 1e-12) for x, y in zip(got, ref))


@pytest.mark.gpu
def test_mixed_and_half_dtypes_return_gradients_in_the_input_dtypes(nfm):
    a, b = _leaf(_a(32, 3, F64, 1)), _leaf(_v((32, 3), 2, torch.float32, 2))
    ga, gb = torch.autograd.grad(nfm.lmdiv(a, b).sum(), (a, b))
    assert ga.dtype == F64 and gb.dtype == torch.float32
    ah, vh = _leaf(_a(32, 3, torch.half, 1)), _leaf(_v(32, 3, torch.half, 2))
    ga, gv = torch.autograd.grad(nfm.batchmatvec(ah, vh).float().sum(), (ah, vh))
    assert ga.dtype == torch.half and gv.dtype == torch.half
    ref = _grads(nfm.batchmatvec, [ah.detach().float(), vh.detach().float()], torch.ones(32, 3, device="cuda"))
    assert _close(ga.float(), ref[0], 1e-3) and _close(gv.float(), ref[1], 1e-3)
    ab = _leaf(_a(32, 3, torch.bfloat16, 1))
    gi, = torch.autograd.grad(nfm.batchinv(ab).sum(), ab)
    gdet, = torch.autograd.grad(nfm.batchdet(ab).sum(), ab)
    assert gi.dtype == torch.bfloat16 and gdet.dtype == torch.bfloat16


@pytest.mark.gpu
def test_backward_follows_a_side_stream_forward(nfm):
    n, B = 4, 200000
    a, b, g = _a(B, n, torch.float32, 1), _v((B, n), 3, torch.float32, 2), _v((B, n), 3, torch.float32, 3)
    ref = _grads(nfm.lmdiv, [a, b], g)
    al, bl = _leaf(a), _leaf(b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        loss = (nfm.lmdiv(al, bl) * g).sum()
    torch.cuda.current_stream().wait_stream(side)
    got = torch.autograd.grad(loss, (al, bl))
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(got, ref))


@pytest.mark.gpu
def test_error_paths(nfm):
    a, b, v = _leaf(_a(4, 3, F64, 1)), _leaf(_v((4, 3), 2, F64, 2)), _leaf(_v(4, 3, F64, 3))
    dev = "cuda"
    with pytest.raises(RuntimeError):
        nfm.batchdet(a, out=torch.empty(4, dtype=F64, device=dev))
    with pytest.raises(RuntimeError):
        nfm.batchinv(a, out=torch.empty(4, 3, 3, dtype=F64, device=dev))
    with pytest.raises(RuntimeError):
        nfm.batchmatvec(a, v, out=torch.empty(4, 3, dtype=F64, device=dev))
    with pytest.raises(RuntimeError):
        nfm.lmdiv(a, b, out=torch.empty(4, 3, 2, dtype=F64, device=dev))
    with pytest.raises(RuntimeError):
        nfm.rmdiv(b.transpose(-1, -2), a, out=torch.empty(4, 2, 3, dtype=F64, device=dev))
    with pytest.raises(RuntimeError):
        nfm.solvevec(a, v, out=torch.empty(4, 3, dtype=F64, device=dev))
    for fn in [lambda: nfm.batchdet(a), lambda: nfm.batchinv(a), lambda: nfm.batchmatvec(a, v), lambda: nfm.lmdiv(a, b),
               lambda: nfm.rmdiv(b.transpose(-1, -2), a), lambda: nfm.inv(a, method="chol")]:
        ga, = torch.autograd.grad(fn().sum(), a, create_graph=True)
        with pytest.raises(RuntimeError):
            torch.autograd.grad(ga.sum(), a)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 6])
def test_no_grad_behaviour_is_unchanged(nfm, n):
    a, b, v = _a(4096, n, torch.float32, 1), _v((4096, n), 3, torch.float32, 2), _v(4096, n, torch.float32, 3)
    r = _v((4096, 2), n, torch.float32, 4)
    calls = [lambda a, b, v, r: nfm.batchdet(a), lambda a, b, v, r: nfm.batchinv(a),
             lambda a, b, v, r: nfm.batchinv(a, method="chol"), lambda a, b, v, r: nfm.batchmatvec(a, v),
             lambda a, b, v, r: nfm.lmdiv(a, b), lambda a, b, v, r: nfm.rmdiv(r, a), lambda a, b, v, r: nfm.inv(a),
             lambda a, b, v, r: nfm.solvevec(a, v), lambda a, b, v, r: nfm.matvec(a, v)]
    for call in calls:
        b0 = _lib.launch_count()
        plain = call(a, b, v, r)
        d_plain = _lib.launch_count() - b0
        leaves = [_leaf(t) for t in (a, b, v, r)]
        with torch.no_grad():
            b0 = _lib.launch_count()
            gated = call(*leaves)
            d_gated = _lib.launch_count() - b0
        assert not plain.requires_grad and not gated.requires_grad
        assert torch.equal(plain, gated) and d_plain == d_gated
