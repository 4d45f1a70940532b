"""Parity of the CUDA path (through the drop-in API -> C ABI) with
(a) the golden fixtures produced by the real reference and (b) the CPU oracle
on seeded inputs.  Metric: worst per-matrix norm-wise relative error; bars are
the north star's 1e-5 (fp32) / 1e-12 (fp64)."""
import pytest
import torch

from conftest import TAGS, TOL
from oracle import generators as G
from oracle import ref_port as P

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.float64]
DEV = "cuda:0"


@pytest.fixture(scope="module")
def nfm():
    import nitorch_fastmath_b200 as pkg
    from nitorch_fastmath_b200 import _lib
    _lib.load()
    return pkg


def close(got, want, dtype, rec=1, scale=1.0):
    assert tuple(got.shape) == tuple(want.shape), (got.shape, want.shape)
    assert got.dtype == want.dtype
    err = G.rel_err(got, want, rec)
    assert err <= TOL[dtype] * scale, f"rel err {err:.3e} > {TOL[dtype] * scale:.1e}"


def close_sum(got, want, terms, dtype):
    """For inp +/- A v the result can cancel to ~0, so the error is measured
    against the size of the terms that were added (backward-error style)."""
    assert tuple(got.shape) == tuple(want.shape) and got.dtype == want.dtype
    num = (got.cpu().double() - want.double()).norm(dim=-1)
    den = sum(t.cpu().double().norm(dim=-1) for t in terms).clamp_min(1e-300)
    err = float((num / den).max()) if num.numel() else 0.0
    assert err <= TOL[dtype], f"rel err {err:.3e} > {TOL[dtype]:.1e}"


# --------------------------------------------------------------------------
# golden fixtures (small batch -> strided kernel)
# --------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_sym_golden(nfm, sym_golden, dtype, n):
    k = f"{TAGS[dtype]}_n{n}"
    mat, vec, inp, reg = (sym_golden(f"{k}_{s}", DEV) for s in ("mat", "vec", "inp", "reg"))
    close(nfm.sym_matvec(mat, vec), sym_golden(f"{k}_matvec"), dtype)
    terms = (sym_golden(f"{k}_inp"), sym_golden(f"{k}_matvec"))
    close_sum(nfm.sym_addmatvec(inp, mat, vec), sym_golden(f"{k}_addmatvec"), terms, dtype)
    close_sum(nfm.sym_submatvec(inp, mat, vec), sym_golden(f"{k}_submatvec"), terms, dtype)
    close(nfm.sym_solve(mat, vec), sym_golden(f"{k}_solve"), dtype)
    close(nfm.sym_solve(mat, vec, reg), sym_golden(f"{k}_solve_reg"), dtype)
    close(nfm.sym_solve(mat, vec, method="lu"), sym_golden(f"{k}_solve"), dtype)
    close(nfm.sym_invert(mat), sym_golden(f"{k}_invert"), dtype)
    close(nfm.sym_invert(mat, True), sym_golden(f"{k}_invert_diag"), dtype)
    close(nfm.sym_invert(mat, method="lu"), sym_golden(f"{k}_invert"), dtype)
    close(nfm.sym_to_full(mat), sym_golden(f"{k}_full"), dtype, 2)
    # symmetric indefinite: closed forms (n <= 4) / pivoted LU (n > 4), as the reference;
    # the default (checked LDL^T, LU fallback per matrix) must agree as well
    ind = sym_golden(f"{k}_ind_mat", DEV)
    close(nfm.sym_solve(ind, vec, method="lu"), sym_golden(f"{k}_ind_solve"), dtype, scale=4)
    close(nfm.sym_solve(ind, vec), sym_golden(f"{k}_ind_solve"), dtype, scale=20)


@pytest.mark.parametrize("dtype", DTYPES)
def test_eps_golden(nfm, sym_golden, dtype):
    t = TAGS[dtype]
    mat, vec = sym_golden(f"{t}_eps2_mat", DEV), sym_golden(f"{t}_eps2_vec", DEV)
    close(nfm.sym_solve(mat, vec, 0.1), sym_golden(f"{t}_eps2_solve"), dtype)
    close(nfm.sym_solve(mat, vec, eps=0.1), sym_golden(f"{t}_eps2_solve"), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_dense_golden(nfm, dense_golden, dtype, n):
    k = f"{TAGS[dtype]}_n{n}"
    a, b, s, rhs = (dense_golden(f"{k}_{x}", DEV) for x in ("a", "b", "spd", "rhs"))
    close(nfm.batchinv(a), dense_golden(f"{k}_inv"), dtype, 2)
    close(nfm.batchinv(a, method="lu"), dense_golden(f"{k}_inv"), dtype, 2)
    close(nfm.batchdet(a), dense_golden(f"{k}_det"), dtype, 0)
    close(nfm.batchmatvec(a, b), dense_golden(f"{k}_matvec"), dtype)
    close(nfm.solvevec(a, b, "lu"), dense_golden(f"{k}_solve_lu"), dtype)
    close(nfm.solvevec(s, b, "chol"), dense_golden(f"{k}_solve_chol"), dtype)
    close(nfm.lmdiv(a, rhs, "lu"), dense_golden(f"{k}_lmdiv_lu"), dtype, 2)
    close(nfm.lmdiv(s, rhs, "chol"), P.lmdiv(s.cpu(), rhs.cpu(), "chol"), dtype, 2)
    close(nfm.inv(s, "chol"), dense_golden(f"{k}_inv_chol"), dtype, 2)
    close(nfm.inv(a, "lu"), dense_golden(f"{k}_inv"), dtype, 2)
    if n in (2, 3):
        # the reference's CUDA closed forms, including det += range * 1e-12
        close(nfm.batchinv(a), dense_golden(f"{k}_closed_inv"), dtype, 2, scale=0.5)
        close(nfm.batchdet(a), dense_golden(f"{k}_closed_det"), dtype, 0)


# --------------------------------------------------------------------------
# seeded batches large enough for the TMA fast path (+ ragged tail)
# --------------------------------------------------------------------------

BATCH = 20011   # prime: full tiles + ragged tail for every tile size


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_sym_fast_path_vs_oracle(nfm, dtype, n):
    from nitorch_fastmath_b200 import _lib
    mat = G.spd_packed(BATCH, n, dtype, seed=n)
    vec = G.vectors(BATCH, n, dtype, seed=50 + n)
    inp = G.vectors(BATCH, n, dtype, seed=90 + n)
    reg = G.vectors(BATCH, n, dtype, seed=70 + n).abs()
    dm, dv, di, dr = (t.to(DEV) for t in (mat, vec, inp, reg))
    x = nfm.sym_solve(dm, dv)
    assert _lib.load().nfm_last_path_was_tma() == 1
    close(x, P.sym_solve(mat, vec), dtype)
    close(nfm.sym_solve(dm, dv, dr), P.sym_solve(mat, vec, reg), dtype)
    close(nfm.sym_solve(dm, dv, 0.25), P.sym_solve(mat, vec, 0.25), dtype)
    close(nfm.sym_solve(dm, dv, [0.5, 0.25][:n]), P.sym_solve(mat, vec, [0.5, 0.25][:n]), dtype)
    close(nfm.sym_solve(dm, dv, method="lu"), P.sym_solve(mat, vec), dtype)
    # the sub-warp cooperative shuffle variant (N >= 5; below it is the closed form)
    close(nfm.sym_solve(dm, dv, method="warp"), P.sym_solve(mat, vec), dtype)
    assert _lib.load().nfm_last_path_was_tma() == (2 if n >= 5 else 1)
    close(nfm.sym_solve(dm, dv, dr, method="warp"), P.sym_solve(mat, vec, reg), dtype)
    close(nfm.sym_matvec(dm, dv), P.sym_matvec(mat, vec), dtype)
    terms = (inp, P.sym_matvec(mat, vec))
    close_sum(nfm.sym_addmatvec(di, dm, dv), P.sym_addmatvec(inp, mat, vec), terms, dtype)
    close_sum(nfm.sym_submatvec(di, dm, dv), P.sym_submatvec(inp, mat, vec), terms, dtype)
    close(nfm.sym_invert(dm), P.sym_invert(mat), dtype)
    close(nfm.sym_invert(dm, True), P.sym_invert(mat, True), dtype)
    close(nfm.sym_invert(dm, method="lu"), P.sym_invert(mat), dtype)
    close(nfm.sym_to_full(dm), P.sym_to_full(mat), dtype, 2)
    close(nfm.sym_det(dm), torch.det(P.sym_to_full(mat.double())).to(dtype), dtype, 0, scale=10)
    close(nfm.sym_outer(dv), P.full_to_sym(vec[..., :, None] * vec[..., None, :]), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_dense_fast_path_vs_oracle(nfm, dtype, n):
    a = G.dense_shifted(BATCH, n, dtype, seed=n)
    b = G.vectors(BATCH, n, dtype, seed=30 + n)
    s = G.dense_spd(BATCH, n, dtype, seed=n)
    da, db, ds = a.to(DEV), b.to(DEV), s.to(DEV)
    # reference CPU branch = LAPACK; n <= 3 on CUDA = closed forms: both must hold
    close(nfm.batchinv(da), P.batchinv(a), dtype, 2)
    close(nfm.batchdet(da), P.batchdet(a), dtype, 0)
    close(nfm.batchmatvec(da, db), P.batchmatvec(a, b), dtype)
    close(nfm.solvevec(da, db), P.solvevec(a, b), dtype)
    close(nfm.solvevec(ds, db, "chol"), P.solvevec(s, b, "chol"), dtype)
    close(nfm.inv(ds, "chol"), P.inv(s, "chol"), dtype, 2)
    if n <= 3:
        close(nfm.batchinv(da), P.closed_inv(a), dtype, 2, scale=0.5)
        close(nfm.batchdet(da), P.closed_det(a), dtype, 0)


@pytest.mark.parametrize("batch", [1, 2, 63, 64, 1023, 1024, 1025, 2 * 1024 + 17, 148 * 1024 + 5])
def test_ragged_tile_boundaries(nfm, batch):
    """Batches around the tile size: full tiles go by TMA, and so does the partial
    last tile (a smaller byte count); only the batch % 4 (% 32 in the segmented layout)
    matrices that break the 16-byte granularity of bulk copies go to the strided
    kernel -- 3x3 fp32, 6x6 fp32, dense 4x4 fp64 (segmented).  All of these batches
    stay below the large-batch switch, so the packed solves run in the small tile
    geometry (3x3: 512-matrix tiles, 6x6: 128); the largest gives each CTA only a few
    tiles.  The large geometry and ring wrap-around are covered by test_steady_state.py."""
    from nitorch_fastmath_b200 import _lib
    for n in (3, 6):
        mat = G.spd_packed(batch, n, torch.float32, seed=batch + n)
        vec = G.vectors(batch, n, torch.float32, seed=batch + n + 1)
        before = _lib.launch_count()
        x = nfm.sym_solve(mat.to(DEV), vec.to(DEV))
        # one launch; the < 4 matrices past the last 16-byte granule take a second, tiny one
        assert _lib.launch_count() - before == (1 if batch % 4 == 0 or batch < 4 else 2)
        assert _lib.load().nfm_last_path_was_tma() == 1
        close(x, P.sym_solve(mat, vec), torch.float32)
        close(nfm.sym_invert(mat.to(DEV)), P.sym_invert(mat), torch.float32)
    a = G.dense_shifted(batch, 4, torch.float64, seed=batch)
    b = G.vectors(batch, 4, torch.float64, seed=batch + 1)
    close(nfm.batchinv(a.to(DEV)), P.batchinv(a), torch.float64, 2)
    close(nfm.batchdet(a.to(DEV)), P.batchdet(a), torch.float64, 0)
    close(nfm.solvevec(a.to(DEV), b.to(DEV)), P.solvevec(a, b), torch.float64)


def _row_permuted(a, seed):
    """Every second matrix gets its rows shuffled: well conditioned, but partial
    pivoting has to exchange rows -- in some lanes of a warp and not in others."""
    g = G.gen(seed)
    a = a.clone()
    n = a.shape[-1]
    for b in range(1, a.shape[0], 2):
        a[b] = a[b][torch.randperm(n, generator=g)]
    return a


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [4, 5, 6, 8, 9, 10])
def test_pivoting_differs_between_lanes_of_a_warp(nfm, dtype, n):
    """The pivoted eliminations skip the row / column exchanges of a step when no
    matrix of the warp needs them (warp vote).  Here half of the lanes need them."""
    batch = 4771 if n >= 8 else 20011        # n >= 8: pool kernel (32-matrix warp tiles) + ragged tile
    a = _row_permuted(G.dense_shifted(batch, n, dtype, seed=n), seed=100 + n)
    b = G.vectors(batch, n, dtype, seed=30 + n)
    da, db = a.to(DEV), b.to(DEV)
    close(nfm.batchinv(da), P.batchinv(a), dtype, 2, scale=4)
    close(nfm.batchdet(da), P.batchdet(a), dtype, 0, scale=4)
    close(nfm.solvevec(da, db), P.solvevec(a, b), dtype, scale=4)
    close(nfm.lmdiv(da, db[..., None].expand(-1, -1, 3).contiguous()),
          P.lmdiv(a, b[..., None].expand(-1, -1, 3).contiguous()), dtype, 2, scale=4)
    # unpermuted input in the same launch shape: no lane exchanges anything
    a0 = G.dense_shifted(batch, n, dtype, seed=n)
    close(nfm.batchinv(a0.to(DEV)), P.batchinv(a0), dtype, 2)
    if n > 4:
        # packed symmetric, method='lu': indefinite matrices pivot, SPD ones do not; interleave them
        m = G.spd_packed(batch, n, dtype, seed=n)
        mi = G.sym_indefinite_packed(batch, n, dtype, seed=n + 1)
        m[1::2] = mi[1::2]
        v = G.vectors(batch, n, dtype, seed=50 + n)
        want = P.sym_solve(m, v)
        close(nfm.sym_solve(m.to(DEV), v.to(DEV), method="lu"), want, dtype, scale=20)
        close(nfm.sym_solve(m.to(DEV), v.to(DEV)), want, dtype, scale=20)
        close(nfm.sym_invert(m.to(DEV), method="lu"), P.sym_invert(m), dtype, scale=20)


@pytest.mark.parametrize("batch", [1, 31, 32, 33, 95, 32 * 148 + 5, 32 * 148 * 3 + 64])
def test_pool_kernel_tile_boundaries(nfm, batch):
    """Heavy ops with large records run on the warp-pool kernel (32-matrix warp
    tiles, buffers handed from warp to warp): batches around the warp tile and
    around one round of the grid.  The largest gives each CTA about three warp
    tiles, fewer than its buffers, so no buffer is refilled here; recycling is
    covered by test_steady_state.py."""
    from nitorch_fastmath_b200 import _lib
    for n, dtype in ((8, torch.float64), (9, torch.float64), (10, torch.float32), (10, torch.float64)):
        a = _row_permuted(G.dense_shifted(batch, n, dtype, seed=batch + n), seed=batch)
        b = G.vectors(batch, n, dtype, seed=batch + 1)
        x = nfm.batchinv(a.to(DEV))
        assert _lib.load().nfm_last_path_was_tma() == 3      # TMA-staged warp-pool kernel
        close(x, P.batchinv(a), dtype, 2, scale=4)
        if dtype == torch.float64:
            # fp64 orders 8..10 invert with TWO lanes per matrix on the pool kernel (16-matrix warp tiles);
            # records spaced wider than their length take the one-thread-per-matrix strided kernel: same bits
            off = torch.empty(batch, n * n + 2, device=DEV, dtype=dtype)[:, :n * n].view(batch, n, n).copy_(a)
            y = nfm.batchinv(off)
            assert _lib.load().nfm_last_path_was_tma() == (0 if batch > 1 else 3)   # one record has no batch stride
            assert torch.equal(x, y)
        close(nfm.batchdet(a.to(DEV)), P.batchdet(a), dtype, 0, scale=4)
        close(nfm.solvevec(a.to(DEV), b.to(DEV)), P.solvevec(a, b), dtype, scale=4)


@pytest.mark.parametrize("batch", [1, 77, 1024, 1030, 5000])
def test_writes_stay_inside_the_output(nfm, batch):
    """compute-sanitizer is not available on the GPU pool, so bounds are checked
    with canaries: outputs live inside a larger buffer whose guard zones must be
    untouched, and inputs must come back bit-identical (TMA bulk stores, the
    segmented layout and the ragged-tail copy all write through raw pointers)."""
    guard = 4096
    sentinel = 12345.0

    def guarded(shape, dtype):
        numel = 1
        for d in shape:
            numel *= d
        buf = torch.full((numel + 2 * guard,), sentinel, device=DEV, dtype=dtype)
        return buf, buf[guard:guard + numel].view(shape)

    def intact(buf, numel):
        return bool((buf[:guard] == sentinel).all()) and bool((buf[guard + numel:] == sentinel).all())

    for dtype in DTYPES:
        for n in (3, 4, 6, 10):
            nn = n * (n + 1) // 2
            mat = G.spd_packed(batch, n, dtype, seed=n).to(DEV)
            vec = G.vectors(batch, n, dtype, seed=n + 1).to(DEV)
            mat0, vec0 = mat.clone(), vec.clone()
            for fn, shape, args in (
                (nfm.sym_solve, (batch, n), (mat, vec)),
                (nfm.sym_matvec, (batch, n), (mat, vec)),
                (nfm.sym_invert, (batch, nn), (mat,)),
            ):
                buf, out = guarded(shape, dtype)
                fn(*args, out=out)
                torch.cuda.synchronize()
                assert intact(buf, out.numel()), (fn.__name__, n, dtype)
                assert not bool((out == sentinel).any())
            if n > 4:
                buf, out = guarded((batch, n), dtype)
                nfm.sym_solve(mat, vec, out=out, method="warp")
                torch.cuda.synchronize()
                assert intact(buf, out.numel())
            assert torch.equal(mat, mat0) and torch.equal(vec, vec0)
        for n in (2, 4, 8, 10):                   # segmented layout; n >= 8: warp-pool kernel
            a = G.dense_shifted(batch, n, dtype, seed=n).to(DEV)
            b = G.vectors(batch, n, dtype, seed=n + 1).to(DEV)
            a0 = a.clone()
            buf, out = guarded((batch, n), dtype)
            nfm.solvevec(a, b, out=out)
            torch.cuda.synchronize()
            assert intact(buf, out.numel()) and not bool((out == sentinel).any())
            buf, out = guarded((batch, n, n), dtype)
            nfm.inv(a, out=out)
            torch.cuda.synchronize()
            assert intact(buf, out.numel()) and not bool((out == sentinel).any())
            assert torch.equal(a, a0)


def test_back_to_back_launches_are_ordered(nfm):
    """Kernels are launched with programmatic stream serialization (they may
    become resident while the previous one drains); a chain of dependent
    in-place calls must still see each other's results."""
    n = 3
    mat = G.spd_packed(300_000, n, torch.float64, seed=1)
    vec = G.vectors(300_000, n, torch.float64, seed=2)
    dm, v = mat.to(DEV), vec.to(DEV)
    for _ in range(8):                      # x <- A^-1 x ; x <- A x   (8 round trips, 16 dependent launches)
        nfm.sym_solve_(dm, v)
        nfm.sym_matvec(dm, v, out=v)
    close(v, vec, torch.float64, scale=100)
    acc = torch.zeros_like(v)
    for _ in range(10):
        nfm.sym_addmatvec_(acc, dm, v)
    close(acc, 10 * P.sym_matvec(mat, vec), torch.float64, scale=100)


# --------------------------------------------------------------------------
# semantics: broadcasting, strides, alignment, dtype, in-place, empty, layouts
# --------------------------------------------------------------------------

@pytest.mark.parametrize("n", [2, 3, 6, 10])
def test_broadcasting(nfm, n):
    dtype = torch.float32
    mat = G.spd_packed((4, 5), n, dtype, seed=1)
    vec = G.vectors((4, 5), n, dtype, seed=2)
    dm, dv = mat.to(DEV), vec.to(DEV)
    # reference behaviour matrix, SURVEY.md appendix A.4
    close(nfm.sym_solve(dm, dv[0, 0]), P.sym_solve(mat, vec[0, 0]), dtype)
    close(nfm.sym_solve(dm[0, 0], dv), P.sym_solve(mat[0, 0], vec), dtype)
    close(nfm.sym_solve(dm[:1], dv), P.sym_solve(mat[:1], vec), dtype)
    close(nfm.sym_solve(dm[:, :1], dv[:1]), P.sym_solve(mat[:, :1], vec[:1]), dtype)
    close(nfm.sym_solve(dm[0, 0], dv[0, 0]), P.sym_solve(mat[0, 0], vec[0, 0]), dtype)
    # superset: unbatched operand in matvec (the reference's own implementation fails there)
    want = P.sym_matvec(mat, vec[0, 0].expand(4, 5, n))
    close(nfm.sym_matvec(dm, dv[0, 0]), want, dtype)
    # large batch with a broadcast operand goes through the TMA path with stride 0
    big_m = G.spd_packed(5000, n, dtype, seed=3)
    v1 = G.vectors(1, n, dtype, seed=4)[0]
    close(nfm.sym_solve(big_m.to(DEV), v1.to(DEV)), P.sym_solve(big_m, v1), dtype)
    big_v = G.vectors(5000, n, dtype, seed=5)
    close(nfm.sym_solve(big_m[0].to(DEV), big_v.to(DEV)), P.sym_solve(big_m[0], big_v), dtype)


@pytest.mark.parametrize("n", [3, 6])
def test_strided_and_unaligned(nfm, n):
    dtype = torch.float32
    nn = n * (n + 1) // 2
    mat = G.spd_packed((7, 900), n, dtype, seed=1)
    vec = G.vectors((7, 900), n, dtype, seed=2)
    dm, dv = mat.to(DEV), vec.to(DEV)
    # transposed batch dims (non-collapsible -> materialised)
    close(nfm.sym_solve(dm.transpose(0, 1), dv.transpose(0, 1)),
          P.sym_solve(mat.transpose(0, 1), vec.transpose(0, 1)), dtype)
    # every second matrix (single non-dense stride -> strided kernel)
    close(nfm.sym_solve(dm[:, ::2], dv[:, ::2]), P.sym_solve(mat[:, ::2], vec[:, ::2]), dtype)
    # storage offset that breaks 16-byte alignment
    flat_m, flat_v = dm.reshape(-1, nn), dv.reshape(-1, n)
    close(nfm.sym_solve(flat_m[1:], flat_v[1:]), P.sym_solve(mat.reshape(-1, nn)[1:], vec.reshape(-1, n)[1:]), dtype)
    # non-unit stride in the coefficient dimension
    wide = torch.zeros(6300, 2 * nn, device=DEV)
    wide[:, ::2] = flat_m
    close(nfm.sym_solve(wide[:, ::2], flat_v), P.sym_solve(mat.reshape(-1, nn), vec.reshape(-1, n)), dtype)
    # coefficient-first storage viewed coefficient-last (what the reference returns, appendix A.4)
    cf = flat_m.t().contiguous().t()
    close(nfm.sym_invert(cf), P.sym_invert(mat.reshape(-1, nn)), dtype)


@pytest.mark.parametrize("n", [3, 6])
def test_coefficient_first_fields_are_read_in_place(nfm, n):
    """Channel-first fields (C, X, Y, Z) viewed coefficient-last -- what nitorch
    keeps and what the reference's own sym_solve returns (_impl/sym.py:398) --
    go to the library with their element stride; no AoS copy is made."""
    from nitorch_fastmath_b200 import _dispatch as D
    dtype = torch.float32
    nn = n * (n + 1) // 2
    shape = (24, 20, 18)
    mat = G.spd_packed(shape, n, dtype, seed=1)
    vec = G.vectors(shape, n, dtype, seed=2)
    mat_cf = mat.to(DEV).movedim(-1, 0).contiguous()       # (NN, X, Y, Z)
    vec_cf = vec.to(DEV).movedim(-1, 0).contiguous()       # (N, X, Y, Z)
    m_view, v_view = mat_cf.movedim(0, -1), vec_cf.movedim(0, -1)
    op = D.as_operand(m_view, shape, 1, dtype, allow_estride=True)
    assert op.ptr == mat_cf.data_ptr() and op.stride == 1 and op.estride == 24 * 20 * 18
    close(nfm.sym_solve(m_view, v_view), P.sym_solve(mat, vec), dtype)
    close(nfm.sym_matvec(m_view, v_view), P.sym_matvec(mat, vec), dtype)
    close(nfm.sym_invert(m_view), P.sym_invert(mat), dtype)
    # mixed: AoS matrix, SoA vector, SoA output written in place
    out_cf = torch.empty_like(vec_cf)
    res = nfm.sym_solve(mat.to(DEV), v_view, out=out_cf.movedim(0, -1))
    assert res.data_ptr() == out_cf.data_ptr()
    close(out_cf.movedim(0, -1), P.sym_solve(mat, vec), dtype)
    # in place on a channel-first field
    nfm.sym_solve_(m_view, v_view)
    close(vec_cf.movedim(0, -1), P.sym_solve(mat, vec), dtype)


def test_dtype_semantics(nfm):
    mat = G.spd_packed(300, 3, torch.float64, seed=1)
    vec = G.vectors(300, 3, torch.float32, seed=2)
    x = nfm.sym_solve(mat.to(DEV), vec.to(DEV))
    assert x.dtype == torch.float32                      # solve -> vec's dtype (reference)
    close(x, P.sym_solve(mat, vec), torch.float32)
    y = nfm.sym_matvec(mat.to(DEV), vec.to(DEV))
    assert y.dtype == torch.float64                      # matvec -> promoted (reference)
    close(y, P.sym_matvec(mat, vec.double()), torch.float64)
    z = nfm.sym_solve(mat.to(DEV), vec.to(DEV), dtype=torch.float64)
    assert z.dtype == torch.float64


def test_half_precision_inputs_follow_reference_dtypes(nfm):
    """fp16 / bf16 are not required (SURVEY 8a) but run through the reference;
    here they compute in fp32 and come back in the reference's result dtype."""
    mat = G.spd_packed(500, 3, torch.float32, seed=1)
    vec = G.vectors(500, 3, torch.float32, seed=2)
    for half in (torch.float16, torch.bfloat16):
        x = nfm.sym_solve(mat.to(DEV, half), vec.to(DEV, half))
        assert x.dtype == half
        want = P.sym_solve(mat.to(half).float(), vec.to(half).float())
        assert G.rel_err(x.float(), want) < (2e-2 if half == torch.bfloat16 else 3e-3)
        assert nfm.sym_matvec(mat.to(DEV, half), vec.to(DEV)).dtype == torch.float32
        assert nfm.sym_invert(mat.to(DEV, half)).dtype == half


def test_cuda_graph_capture(nfm):
    """The C ABI neither allocates nor synchronises, so calls can be captured
    in a CUDA graph and replayed (launch-bound loops, DESIGN.md section 3.1)."""
    mat = G.spd_packed(100_000, 3, torch.float32, seed=1)
    vec = G.vectors(100_000, 3, torch.float32, seed=2)
    dm, dv = mat.to(DEV), vec.to(DEV)
    out = torch.empty_like(dv)
    nfm.sym_solve(dm, dv, out=out)                      # warm (function attributes, occupancy)
    torch.cuda.synchronize()
    out.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(4):
            nfm.sym_solve(dm, dv, out=out)
    assert float(out.abs().sum()) == 0.0                # captured, not run
    graph.replay()
    torch.cuda.synchronize()
    close(out, P.sym_solve(mat, vec), torch.float32)


@pytest.mark.parametrize("n", [3, 6])
def test_inplace_variants(nfm, n):
    dtype = torch.float32
    mat = G.spd_packed(9000, n, dtype, seed=1)
    vec = G.vectors(9000, n, dtype, seed=2)
    inp = G.vectors(9000, n, dtype, seed=3)
    dm = mat.to(DEV)
    v = vec.to(DEV)
    r = nfm.sym_solve_(dm, v)
    assert r.data_ptr() == v.data_ptr()
    close(v, P.sym_solve(mat, vec), dtype)
    i = inp.to(DEV)
    terms = (inp, P.sym_matvec(mat, vec))
    assert nfm.sym_addmatvec_(i, dm, vec.to(DEV)).data_ptr() == i.data_ptr()
    close_sum(i, P.sym_addmatvec(inp, mat, vec), terms, dtype)
    i = inp.to(DEV)
    nfm.sym_submatvec_(i, dm, vec.to(DEV))
    close_sum(i, P.sym_submatvec(inp, mat, vec), terms, dtype)
    m2 = mat.to(DEV)
    assert nfm.sym_invert_(m2).data_ptr() == m2.data_ptr()
    close(m2, P.sym_invert(mat), dtype)
    out = torch.empty(9000, n, device=DEV)
    assert nfm.sym_solve(dm, vec.to(DEV), out=out) is out
    close(out, P.sym_solve(mat, vec), dtype)


def test_empty_and_unbatched(nfm):
    mat = G.spd_packed((0, 5), 3, torch.float32)
    vec = G.vectors((0, 5), 3, torch.float32)
    assert tuple(nfm.sym_solve(mat.to(DEV), vec.to(DEV)).shape) == (0, 5, 3)
    assert tuple(nfm.sym_invert(mat.to(DEV)).shape) == (0, 5, 6)
    assert tuple(nfm.batchinv(torch.zeros(0, 4, 4, device=DEV)).shape) == (0, 4, 4)
    m1 = G.spd_packed(1, 3, torch.float32)[0]
    v1 = G.vectors(1, 3, torch.float32)[0]
    close(nfm.sym_solve(m1.to(DEV), v1.to(DEV)), P.sym_solve(m1, v1), torch.float32)


@pytest.mark.parametrize("n", [1, 2, 3, 5])
def test_compact_layouts(nfm, n):
    """scaled identity / diagonal / full layouts (reference sym.py:16-24)."""
    dtype = torch.float64
    vec = G.vectors(3000, n, dtype, seed=2)
    dv = vec.to(DEV)
    sc = 1 + G.vectors(3000, 1, dtype, seed=3).abs()
    dg = 1 + G.vectors(3000, n, dtype, seed=4).abs()
    full = P.sym_to_full(G.spd_packed(3000, n, dtype, seed=5))
    if n > 1:
        close(nfm.sym_matvec(sc.to(DEV), dv), sc * vec, dtype)
        close(nfm.sym_solve(sc.to(DEV), dv), vec / sc, dtype)
        close(nfm.sym_matvec(dg.to(DEV), dv), dg * vec, dtype)
        close(nfm.sym_solve(dg.to(DEV), dv), vec / dg, dtype)
        close(nfm.sym_solve(dg.to(DEV), dv, 0.5), vec / (dg + 0.5), dtype)
        flat = full.reshape(3000, n * n)
        close(nfm.sym_matvec(flat.to(DEV), dv), P.batchmatvec(full, vec), dtype)
        close(nfm.sym_solve(flat.to(DEV), dv), P.solvevec(full, vec), dtype)


@pytest.mark.parametrize("n", [5, 6, 8, 10])
def test_indefinite_and_zero_pivot_matrices_default_method(nfm, n):
    """The reference solves any invertible symmetric matrix of order > 4 (pivoted
    LU).  Plain LDL^T breaks on a zero leading pivot; the default method detects
    it per matrix and falls back, `method='ldl'` does not."""
    dtype = torch.float64
    batch = 4096
    ind = G.sym_indefinite_packed(batch, n, dtype, seed=n)
    vec = G.vectors(batch, n, dtype, seed=n + 1)
    want = P.sym_solve(ind, vec)
    close(nfm.sym_solve(ind.to(DEV), vec.to(DEV)), want, dtype, scale=1e3)
    inv_want = P.sym_invert(ind)
    close(nfm.sym_invert(ind.to(DEV)), inv_want, dtype, scale=1e3)
    # a_00 = 0 exactly: [[0, 1], [1, 0]] (+) I
    hard = torch.zeros(batch, n * (n + 1) // 2, dtype=dtype)
    hard[:, 1:n] = 1.0
    hard[:, n] = 1.0          # a_01
    want = P.sym_solve(hard, vec)
    got = nfm.sym_solve(hard.to(DEV), vec.to(DEV))
    close(got, want, dtype, scale=10)
    bad = nfm.sym_solve(hard.to(DEV), vec.to(DEV), method="ldl")
    assert not torch.isfinite(bad).all()


def test_singular_does_not_trap(nfm):
    # reference: closed forms give NaN/inf for singular input, no exception (appendix A.4)
    x = nfm.sym_solve(torch.zeros(64, 6, device=DEV), torch.ones(64, 3, device=DEV))
    assert not torch.isfinite(x).any()
    x = nfm.sym_solve(torch.zeros(64, 21, device=DEV), torch.ones(64, 6, device=DEV))
    assert not torch.isfinite(x).any()
    torch.cuda.synchronize()


@pytest.mark.parametrize("dtype", DTYPES)
def test_next_rows_golden(nfm, extra_golden, dtype):
    """sym_outer / sym_matmul against outputs of the real reference (incl. its
    J H J^T behaviour for k == d <= 3)."""
    t = TAGS[dtype]
    for n in (1, 2, 3, 5, 10):
        close(nfm.sym_outer(extra_golden(f"{t}_outer{n}_x", DEV)), extra_golden(f"{t}_outer{n}"), dtype)
    for k, d in ((1, 1), (2, 2), (3, 3), (4, 4), (2, 3), (4, 2), (3, 1), (5, 3), (6, 6)):
        got = nfm.sym_matmul(extra_golden(f"{t}_jhj{k}x{d}_j", DEV), extra_golden(f"{t}_jhj{k}x{d}_h", DEV))
        close(got, extra_golden(f"{t}_jhj{k}x{d}"), dtype)


def test_sym_matmul(nfm):
    dtype = torch.float64
    for k, d in [(1, 1), (2, 2), (3, 3), (4, 4), (2, 3), (4, 2), (3, 1), (6, 6), (5, 3), (3, 7), (10, 10)]:
        j = G.vectors((2000, k), d, dtype, seed=k * 10 + d)
        h = G.spd_packed(2000, k, dtype, seed=k)
        hf = P.sym_to_full(h)
        if k == d and k <= 3:      # the reference's unrolled branches: J H J^T
            want = j @ hf @ j.transpose(-1, -2)
        else:                      # documented: J^T H J
            want = j.transpose(-1, -2) @ hf @ j
        close(nfm.sym_matmul(j.to(DEV), h.to(DEV)), P.full_to_sym(want), dtype)


# --------------------------------------------------------------------------
# the reference's own tests/test_batched.py, run on CUDA against this package
# --------------------------------------------------------------------------

def test_reference_test_batchmatvec(nfm):
    def check(mat, vec):
        return torch.allclose(nfm.batchmatvec(mat, vec), mat.matmul(vec.unsqueeze(-1)).squeeze(-1))
    g = torch.Generator(device=DEV).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    assert check(r(2, 1, 1), r(2, 2, 1)), "1x1"
    assert check(r(2, 2, 2), r(2, 2, 2)), "2x2"
    assert check(r(2, 3, 3), r(2, 2, 3)), "3x3"
    assert check(r(2, 4, 5), r(2, 2, 5)), "4x5"
    assert check(r(2, 2, 4, 5), r(5)), "mat longer"


def test_reference_test_batchdet_and_inv(nfm):
    """tests/test_batched.py:44-97 of the reference at ITS tolerance (default allclose:
    rtol 1e-5, atol 1e-8, fp32, against torch on the same device).  The reference draws
    unseeded randn(2, n, n); two different fp32 algorithms cannot agree to 1e-5 on a
    nearly singular draw, so here ten seeded draws are made and those with a condition
    number below 30 (most of them) must pass -- at least half of the draws are checked."""
    checked = 0
    for seed in range(10):
        g = torch.Generator(device=DEV).manual_seed(seed)
        for n in (1, 2, 3, 4):
            mat = torch.randn(2, n, n, device=DEV, generator=g)
            if float(torch.linalg.cond(mat.double()).max()) < 30:
                checked += 1
                assert torch.allclose(nfm.batchdet(mat), torch.det(mat)), (seed, n)
            mat.diagonal(0, -1, -2).add_(10)
            assert torch.allclose(nfm.batchinv(mat), torch.linalg.inv(mat)), (seed, n)
    assert checked >= 20, checked


# --------------------------------------------------------------------------
# full-size properties (BASELINE.json configs) -- size-independent checks
# --------------------------------------------------------------------------

def _device_spd(batch, n, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randn(batch, n, n, device=DEV, dtype=dtype, generator=g)
    full = a @ a.transpose(-1, -2)
    full.diagonal(0, -1, -2).add_(n)
    iu = torch.triu_indices(n, n, 1, device=DEV)
    return torch.cat([full.diagonal(0, -1, -2), full[..., iu[0], iu[1]]], -1).contiguous()


@pytest.mark.parametrize("n,side", [(3, 256), (6, 192), (10, 160)])
def test_full_size_round_trip(nfm, n, side):
    """config 2 / 3 / 5: solve then matvec returns the right-hand side;
    invert(invert(A)) == A; the solve is linear in the right-hand side."""
    dtype = torch.float32
    batch = side ** 3
    mat = _device_spd(batch, n, dtype, seed=n)
    g = torch.Generator(device=DEV).manual_seed(99)
    vec = torch.randn(batch, n, device=DEV, dtype=dtype, generator=g)
    x = nfm.sym_solve(mat, vec)
    back = nfm.sym_matvec(mat, x)
    err = ((back - vec).norm(dim=-1) / vec.norm(dim=-1)).max().item()
    assert err < 2e-5, err
    x2 = nfm.sym_solve(mat, 2 * vec)
    assert ((x2 - 2 * x).norm(dim=-1) / x.norm(dim=-1)).max().item() < 1e-6
    # slab parity against the oracle on a slice the CPU finishes in seconds
    sl = slice(batch // 2, batch // 2 + (50000 if n <= 6 else 20000))
    want = P.sym_solve(mat[sl].cpu(), vec[sl].cpu())
    close(x[sl], want, dtype)
    if n > 4:
        # the north star's nominal path for N > 4 (sub-warp shuffle kernel) and pivoted LU, at full size
        xw = nfm.sym_solve(mat, vec, method="warp")
        assert ((xw - x).norm(dim=-1) / x.norm(dim=-1)).max().item() < 5e-6
        close(xw[sl], want, dtype)
        xl = nfm.sym_solve(mat, vec, method="lu")
        assert ((xl - x).norm(dim=-1) / x.norm(dim=-1)).max().item() < 5e-6
        del xw, xl
    inv = nfm.sym_invert(mat)
    again = nfm.sym_invert(inv)
    assert ((again - mat).norm(dim=-1) / mat.norm(dim=-1)).max().item() < 5e-5
    isl = slice(batch // 2, batch // 2 + (50000 if n <= 6 else 4000))    # the reference inverts with N solves: slow on the CPU
    close(inv[isl], P.sym_invert(mat[isl].cpu()), dtype)


def test_config4_dense_fp64(nfm):
    """config 4 (general 4x4 fp64) at its full size, 64 Mi matrices (8.6 GB in, 8.6 GB out):
    A A^-1 = I, det(A^-1) = 1/det(A), solve residual, oracle on slices."""
    n, batch = 4, 64 << 20
    g = torch.Generator(device=DEV).manual_seed(4)
    a = torch.randn(batch, n, n, device=DEV, dtype=torch.float64, generator=g)
    a.diagonal(0, -1, -2).add_(10)
    b = torch.randn(batch, n, device=DEV, dtype=torch.float64, generator=g)
    inv = nfm.batchinv(a)
    eye = torch.eye(n, device=DEV, dtype=torch.float64)
    worst = 0.0
    for c in range(0, batch, 8 << 20):                      # in chunks: a @ inv of the whole batch would take 8.6 GB more
        worst = max(worst, (a[c:c + (8 << 20)] @ inv[c:c + (8 << 20)] - eye).abs().max().item())
    assert worst < 1e-13, worst
    d, di = nfm.batchdet(a), nfm.batchdet(inv)
    assert (d * di - 1).abs().max().item() < 1e-12
    x = nfm.solvevec(a, b)
    worst = 0.0
    for c in range(0, batch, 8 << 20):
        worst = max(worst, ((a[c:c + (8 << 20)] @ x[c:c + (8 << 20), :, None])[..., 0] - b[c:c + (8 << 20)]).abs().max().item())
    assert worst < 1e-12, worst
    for start in (12345, batch // 2 + 7, batch - 100000):   # first slab, middle, the very end
        sl = slice(start, start + 100000)
        close(inv[sl], P.batchinv(a[sl].cpu()), torch.float64, 2)
        close(d[sl], P.batchdet(a[sl].cpu()), torch.float64, 0)
        close(x[sl], P.solvevec(a[sl].cpu(), b[sl].cpu()), torch.float64)


# --------------------------------------------------------------------------
# host-resident operands: the chunked H2D / kernel / D2H pipeline
# --------------------------------------------------------------------------

@pytest.mark.parametrize("n", [3, 6])
def test_host_pipeline(nfm, n):
    dtype = torch.float32
    batch = 1_000_003
    mat = G.spd_packed(batch, n, dtype, seed=1).pin_memory()
    vec = G.vectors(batch, n, dtype, seed=2).pin_memory()
    x = nfm.sym_solve(mat, vec)
    assert x.device.type == "cpu"
    xd = nfm.sym_solve(mat.to(DEV), vec.to(DEV)).cpu()
    assert torch.equal(x, xd)
    sl = slice(500_000, 520_000)
    close(x[sl], P.sym_solve(mat[sl], vec[sl]), dtype)
    inv = nfm.sym_invert(mat)
    assert torch.equal(inv, nfm.sym_invert(mat.to(DEV)).cpu())
    y = nfm.sym_matvec(mat, vec)
    assert torch.equal(y, nfm.sym_matvec(mat.to(DEV), vec.to(DEV)).cpu())
    # non-plain host operands take the whole-upload path
    close(nfm.sym_solve(mat[:1000, :], vec[0]), P.sym_solve(mat[:1000], vec[0]), dtype)


@pytest.mark.parametrize("n,dtype", [(4, torch.float64), (3, torch.float32), (8, torch.float64)])
def test_host_pipeline_dense(nfm, n, dtype):
    """CPU operands of the dense routines are streamed through the GPU in chunks
    (nfm_batch_*_host): same bits as the device call, results on the CPU."""
    batch = 300_007
    a = G.dense_shifted(batch, n, dtype, seed=n).pin_memory()
    b = G.vectors(batch, n, dtype, seed=n + 1).pin_memory()
    b3 = G.vectors((batch, n), 3, dtype, seed=n + 2).pin_memory()
    da, db, db3 = a.to(DEV), b.to(DEV), b3.to(DEV)
    inv = nfm.batchinv(a)
    assert inv.device.type == "cpu" and torch.equal(inv, nfm.batchinv(da).cpu())
    assert torch.equal(nfm.batchdet(a), nfm.batchdet(da).cpu())
    x = nfm.solvevec(a, b)
    assert x.device.type == "cpu" and torch.equal(x, nfm.solvevec(da, db).cpu())
    assert torch.equal(nfm.lmdiv(a, b3), nfm.lmdiv(da, db3).cpu())
    out = torch.empty_like(b).pin_memory()
    assert nfm.solvevec(a, b, out=out).data_ptr() == out.data_ptr() and torch.equal(out, x)
    sl = slice(150_000, 152_000)
    close(x[sl], P.solvevec(a[sl], b[sl]), dtype)
    close(inv[sl], P.batchinv(a[sl]), dtype, 2)
    # non-plain host operands (a strided view) take the whole-upload path
    close(nfm.batchinv(a[::7]), P.batchinv(a[::7]), dtype, 2)


def test_single_process_multi_gpu_host_sharding(nfm):
    """nitorch_fastmath_b200.multi_gpu: one process, the batch cut into slabs,
    one host pipeline per device (all visible devices; 1 on a single-GPU box)."""
    from nitorch_fastmath_b200 import multi_gpu
    n, batch = 3, 3_000_017
    mat = G.spd_packed(batch, n, torch.float32, seed=1).pin_memory()
    vec = G.vectors(batch, n, torch.float32, seed=2).pin_memory()
    x = multi_gpu.sym_solve_multi(mat, vec)
    ref = nfm.sym_solve(mat.to(DEV), vec.to(DEV)).cpu()
    assert torch.equal(x, ref)                                  # slabs are independent: bit-identical
    sl = slice(batch // 2 - 5000, batch // 2 + 5000)            # straddles the 2-GPU slab boundary
    close(x[sl], P.sym_solve(mat[sl], vec[sl]), torch.float32)
    assert torch.equal(multi_gpu.sym_invert_multi(mat), nfm.sym_invert(mat.to(DEV)).cpu())
    assert torch.equal(multi_gpu.sym_matvec_multi(mat, vec), nfm.sym_matvec(mat.to(DEV), vec.to(DEV)).cpu())
    if torch.cuda.device_count() > 1:
        assert torch.equal(multi_gpu.sym_solve_multi(mat, vec, devices=[1]), ref)


def _random_view(t, rng):
    """A random view / re-layout of ``t`` with the same values and shape."""
    kind = rng.choice(["plain", "channel_first", "sliced", "transposed_batch", "offset", "double"])
    if kind == "channel_first":
        return t.movedim(-1, 0).contiguous().movedim(0, -1)
    if kind == "sliced":                       # every second element of a wider buffer
        wide = torch.zeros(*t.shape[:-1], 2 * t.shape[-1], device=t.device, dtype=t.dtype)
        wide[..., ::2] = t
        return wide[..., ::2]
    if kind == "transposed_batch" and t.dim() >= 3:
        return t.transpose(0, 1).contiguous().transpose(0, 1)
    if kind == "offset":                       # storage offset that breaks 16-byte alignment
        flat = torch.zeros(t.numel() + 1, device=t.device, dtype=t.dtype)
        flat[1:] = t.reshape(-1)
        return flat[1:].view(t.shape)
    if kind == "double":
        return t.double()
    return t


def test_randomised_shapes_views_and_broadcasting(nfm):
    """60 seeded random cases: order, batch shape, which operand is broadcast,
    memory layout of every operand, regulariser kind -- all against the oracle."""
    import random
    rng = random.Random(1234)
    for case in range(60):
        n = rng.randint(1, 10)
        nb = rng.randint(1, 3)
        batch = tuple(rng.choice([1, 2, 3, 5, 17, 64]) for _ in range(nb))
        if rng.random() < 0.25:
            batch = (rng.choice([700, 1500, 4099]),)         # long enough for TMA tiles + ragged tail
        mat = G.spd_packed(batch, n, torch.float32, seed=case)
        vec = G.vectors(batch, n, torch.float32, seed=1000 + case)
        # broadcast one operand along a random subset of batch dims
        if rng.random() < 0.4:
            which = rng.choice(["mat", "vec"])
            idx = tuple(slice(0, 1) if rng.random() < 0.6 else slice(None) for _ in batch)
            if which == "mat":
                mat = mat[idx]
            else:
                vec = vec[idx]
        reg_kind = rng.choice([None, None, "scalar", "vector", "field"])
        reg = {None: None, "scalar": 0.3, "vector": [0.5, 0.1][:min(n, 2)],
               "field": G.vectors(torch.broadcast_shapes(mat.shape[:-1], vec.shape[:-1]), n, torch.float32, seed=case).abs()}[reg_kind]
        want = P.sym_solve(mat, vec, reg)
        dm, dv = _random_view(mat.to(DEV), rng), _random_view(vec.to(DEV), rng)
        dr = reg.to(DEV) if torch.is_tensor(reg) else reg
        got = nfm.sym_solve(dm, dv, dr)
        tol_dtype = torch.float32
        assert tuple(got.shape) == tuple(want.shape), (case, got.shape, want.shape)
        err = G.rel_err(got, want)
        assert err <= TOL[tol_dtype], (case, n, batch, err)
        # matvec of the solution gives the right-hand side back (shape semantics of matvec)
        full_mat = mat.expand(*want.shape[:-1], mat.shape[-1])
        if reg is None:
            back = nfm.sym_matvec(_random_view(full_mat.contiguous().to(DEV), rng), got)
            assert G.rel_err(back, vec.expand_as(want)) <= 5e-5, (case, n)
        inv = nfm.sym_invert(_random_view(mat.to(DEV), rng))
        assert G.rel_err(inv, P.sym_invert(mat)) <= TOL[torch.float32], (case, n)


def test_sugar_surface(nfm):
    """lmdiv / rmdiv / inv / solvevec / matvec with `out=` and both methods
    (reference sugar.py:75-341)."""
    dtype = torch.float64
    for n in (2, 3, 5, 8):
        a = G.dense_shifted((6, 50), n, dtype, seed=n)
        spd = G.dense_spd((6, 50), n, dtype, seed=n)
        b = G.vectors((6, 50, 4), n, dtype, seed=n + 1)              # (…, k=4, n): right-division operand
        rhs = b.transpose(-1, -2).contiguous()                        # (…, n, k)
        da, ds, db, dr = a.to(DEV), spd.to(DEV), b.to(DEV), rhs.to(DEV)
        close(nfm.lmdiv(da, dr), torch.linalg.solve(a, rhs), dtype, 2)
        close(nfm.lmdiv(ds, dr, method="chol"), torch.linalg.solve(spd, rhs), dtype, 2)
        close(nfm.rmdiv(db, da), b @ torch.linalg.inv(a), dtype, 2, scale=10)
        out = torch.empty(6, 50, n, 4, device=DEV, dtype=dtype)
        assert nfm.lmdiv(da, dr, out=out) is out
        close(out, torch.linalg.solve(a, rhs), dtype, 2)
        vec = G.vectors((6, 50), n, dtype, seed=n + 2)
        o1 = torch.empty(6, 50, n, device=DEV, dtype=dtype)
        assert nfm.solvevec(da, vec.to(DEV), out=o1).data_ptr() == o1.data_ptr()   # a squeezed view of out, as the reference
        close(o1, P.solvevec(a, vec), dtype)
        o2 = torch.empty(6, 50, n, device=DEV, dtype=dtype)
        nfm.matvec(da, vec.to(DEV), out=o2)
        close(o2, P.batchmatvec(a, vec), dtype)
        o3 = torch.empty(6, 50, n, n, device=DEV, dtype=dtype)
        nfm.inv(ds, "chol", out=o3)
        close(o3, torch.linalg.inv(spd), dtype, 2)
    with pytest.raises(NotImplementedError):
        nfm.lmdiv(torch.zeros(3, 4, 5, device=DEV), torch.zeros(3, 4, 1, device=DEV))
    with pytest.raises(NotImplementedError):
        nfm.inv(torch.eye(3, device=DEV)[None], method="svd")


def test_tensors_on_a_non_current_device(nfm):
    """Operands on cuda:1 while cuda:0 is current: the call must run on the
    tensors' device (needs a 2-GPU box; skipped otherwise)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    assert torch.cuda.current_device() == 0
    d1 = torch.device("cuda:1")
    for n in (3, 6):
        mat = G.spd_packed(50_000, n, torch.float32, seed=n)
        vec = G.vectors(50_000, n, torch.float32, seed=n + 1)
        x = nfm.sym_solve(mat.to(d1), vec.to(d1))
        assert x.device == d1
        close(x, P.sym_solve(mat, vec), torch.float32)
        close(nfm.sym_solve(mat.to(d1)[::2], vec.to(d1)[::2]), P.sym_solve(mat[::2], vec[::2]), torch.float32)
        close(nfm.sym_invert(mat.to(d1)), P.sym_invert(mat), torch.float32)
        a = G.dense_shifted(10_000, n, torch.float64, seed=n)
        close(nfm.batchinv(a.to(d1)), P.batchinv(a), torch.float64, 2)
    with pytest.raises(RuntimeError):
        nfm.sym_solve(mat.to(d1), vec.to("cuda:0"))
    assert torch.cuda.current_device() == 0


def test_randomised_dense_shapes_and_views(nfm):
    """40 seeded random cases for the dense routines: order, batch shape, dtype,
    non-contiguous / broadcast operands -- against the oracle (LAPACK)."""
    import random
    rng = random.Random(4321)
    for case in range(40):
        n = rng.randint(1, 10)
        dtype = rng.choice(DTYPES)
        nb = rng.randint(1, 3)
        batch = tuple(rng.choice([1, 2, 3, 7, 33]) for _ in range(nb))
        if rng.random() < 0.25:
            batch = (rng.choice([300, 1100, 2053]),)
        a = G.dense_shifted(batch, n, dtype, seed=case)
        b = G.vectors(batch, n, dtype, seed=500 + case)
        da, db = a.to(DEV), b.to(DEV)
        layout = rng.choice(["plain", "transposed_storage", "sliced", "offset"])
        if layout == "transposed_storage":      # column-major storage viewed row-major
            da = da.transpose(-1, -2).contiguous().transpose(-1, -2)
        elif layout == "sliced":
            wide = torch.zeros(*batch, n, 2 * n, device=DEV, dtype=dtype)
            wide[..., ::2] = da
            da = wide[..., ::2]
        elif layout == "offset":
            flat = torch.zeros(da.numel() + 1, device=DEV, dtype=dtype)
            flat[1:] = da.reshape(-1)
            da = flat[1:].view(da.shape)
        close(nfm.batchinv(da), P.batchinv(a), dtype, 2)
        close(nfm.batchdet(da), P.batchdet(a), dtype, 0)
        close(nfm.solvevec(da, db), P.solvevec(a, b), dtype)
        close(nfm.batchmatvec(da, db), P.batchmatvec(a, b), dtype)
        # vector broadcast against the batch of matrices
        close(nfm.batchmatvec(da, db.reshape(-1, n)[0]), P.batchmatvec(a, b.reshape(-1, n)[0]), dtype)
        close(nfm.solvevec(da, db.reshape(-1, n)[0].expand(*batch, n)), P.solvevec(a, b.reshape(-1, n)[0].expand(*batch, n)), dtype)
        k = rng.randint(2, 6)
        rhs = G.vectors((*batch, n), k, dtype, seed=900 + case)
        close(nfm.lmdiv(da, rhs.to(DEV)), P.lmdiv(a, rhs), dtype, 2)


def _per_matrix_err(x, ref):
    x, ref = x.detach().cpu().double(), ref.detach().cpu().double()
    return (x - ref).norm(dim=-1) / ref.norm(dim=-1).clamp_min(1e-300)


@pytest.mark.parametrize("n", [2, 3, 4, 6, 10])
def test_accuracy_tracks_the_reference_on_ill_conditioned_spd(nfm, n):
    """Beyond the well-conditioned generator of the north star: SPD matrices with
    condition number 1e3 in fp32.  Neither implementation can meet 1e-5 there;
    what must hold is that this path is not less accurate than the reference's
    CPU path (both measured against an fp64 solve)."""
    batch = 20_000
    g = G.gen(100 + n)
    q, _ = torch.linalg.qr(torch.randn(batch, n, n, dtype=torch.float64, generator=g))
    lam = torch.exp(torch.rand(batch, n, dtype=torch.float64, generator=g) * (-6.9))      # in (1e-3, 1]
    full = (q * lam[..., None, :]) @ q.transpose(-1, -2)
    mat64 = P.full_to_sym(full)
    vec64 = torch.randn(batch, n, dtype=torch.float64, generator=g)
    truth = torch.linalg.solve(full, vec64[..., None])[..., 0]
    mat, vec = mat64.float(), vec64.float()
    e_ref = _per_matrix_err(P.sym_solve(mat, vec), truth)
    e_ours = _per_matrix_err(nfm.sym_solve(mat.to(DEV), vec.to(DEV)), truth)
    # medians within 2x, tails within 4x of the reference's own error
    assert e_ours.median() <= 2 * e_ref.median() + 1e-7, (float(e_ours.median()), float(e_ref.median()))
    assert e_ours.quantile(0.99) <= 4 * e_ref.quantile(0.99) + 1e-6
    assert torch.isfinite(e_ours).all()
    # fp64 on the same matrices stays at rounding level
    e64 = _per_matrix_err(nfm.sym_solve(mat64.to(DEV), vec64.to(DEV)), truth)
    assert e64.max() < 1e-9


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [1, 2, 3, 4, 6, 10])
def test_fused_solve_update(nfm, dtype, n):
    """x - alpha (A + lam I)^-1 v in one pass == the chain sym_solve -> update (oracle)."""
    batch = 30_011
    mat = G.spd_packed(batch, n, dtype, seed=n)
    vec = G.vectors(batch, n, dtype, seed=n + 1)
    x = G.vectors(batch, n, dtype, seed=n + 2)
    for lam, alpha in ((0.0, 1.0), (0.3, 0.5)):
        step = P.sym_solve(mat, vec, lam if lam else None)
        want = x - alpha * step
        got = nfm.sym_solve_update(x.to(DEV), mat.to(DEV), vec.to(DEV), lam, alpha)
        num = (got.cpu().double() - want.double()).norm(dim=-1)
        den = (x.double().norm(dim=-1) + alpha * step.double().norm(dim=-1)).clamp_min(1e-300)
        assert float((num / den).max()) <= TOL[dtype]
    xd = x.to(DEV)
    assert nfm.sym_solve_update_(xd, mat.to(DEV), vec.to(DEV), 0.3, 0.5).data_ptr() == xd.data_ptr()
    num = (xd.cpu().double() - want.double()).norm(dim=-1)
    assert float((num / den).max()) <= TOL[dtype]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [2, 3, 6, 10])
def test_fused_solve_update_per_voxel_regulariser(nfm, dtype, n):
    """The reference's documented regulariser (_impl/sym.py:356-357) as a fourth staged
    operand of the fused update: x - alpha (A + lam I + diag(d))^-1 v  ==  the oracle chain."""
    batch = 30_011
    mat = G.spd_packed(batch, n, dtype, seed=n)
    vec = G.vectors(batch, n, dtype, seed=n + 1)
    x = G.vectors(batch, n, dtype, seed=n + 2)
    reg = G.vectors(batch, n, dtype, seed=n + 3).abs()
    lam, alpha = 0.25, 0.5
    step = P.sym_solve(mat, vec, reg + lam)
    want = x - alpha * step
    den = (x.double().norm(dim=-1) + alpha * step.double().norm(dim=-1)).clamp_min(1e-300)
    dm, dv, dx, dr = (t.to(DEV) for t in (mat, vec, x, reg))
    for kw in (dict(diag=dr), dict(diag=dr[:1].expand(batch, n) * 0 + dr), dict(diag=dr, out=torch.empty_like(dx))):
        got = nfm.sym_solve_update(dx, dm, dv, lam, alpha, **kw)
        assert float(((got.cpu().double() - want.double()).norm(dim=-1) / den).max()) <= TOL[dtype]
    # one (n,) regulariser broadcast to the whole field, and a shape-(1,) tensor
    r1 = reg[0]
    want1 = x - alpha * P.sym_solve(mat, vec, r1 + lam)
    got1 = nfm.sym_solve_update(dx, dm, dv, lam, alpha, diag=r1.to(DEV))
    assert float(((got1.cpu().double() - want1.double()).norm(dim=-1) / den).max()) <= TOL[dtype] * 2
    close(nfm.sym_solve(dm, dv, torch.tensor([0.125], device=DEV, dtype=dtype)), P.sym_solve(mat, vec, 0.125), dtype)
    strided = torch.arange(2 * n, device=DEV, dtype=dtype)[::2] * 0.01 + 0.1       # ADVICE r1: non-contiguous 1-D diag
    close(nfm.sym_solve(dm, dv, strided), P.sym_solve(mat, vec, strided.cpu()), dtype)
    xd = dx.clone()
    assert nfm.sym_solve_update_(xd, dm, dv, lam, alpha, diag=dr).data_ptr() == xd.data_ptr()
    assert float(((xd.cpu().double() - want.double()).norm(dim=-1) / den).max()) <= TOL[dtype]


@pytest.mark.parametrize("dtype", DTYPES)
def test_fused_matmul_solve(nfm, dtype):
    """(J^T H J + diag(d))^-1 g built and solved in registers == the oracle chain
    sym_matmul -> sym_solve (reference _impl/sym.py:637-670 then :327-398), including
    the reference's J H J^T for k == d <= 3."""
    batch = 20_011
    for k, d in [(1, 1), (2, 2), (3, 3), (4, 4), (6, 6), (2, 3), (3, 2), (4, 3), (6, 3), (3, 6), (5, 6), (6, 5), (8, 3), (10, 3), (10, 2), (7, 1)]:
        j = G.vectors((batch, k), d, dtype, seed=k * 10 + d)
        j = 0.3 * j + 2 * torch.eye(k, d, dtype=dtype)    # singular values in about [1, 3]: J^T H J well conditioned when k >= d
        h = G.spd_packed(batch, k, dtype, seed=k)
        g = G.vectors(batch, d, dtype, seed=k + d)
        reg = G.vectors(batch, d, dtype, seed=k + d + 1).abs() + (1.0 if k < d else 0.0)   # k < d: J^T H J is singular
        a = P.sym_matmul(j, h)
        dj, dh, dg, dr = (t.to(DEV) for t in (j, h, g, reg))
        close(nfm.sym_matmul(dj, dh), a, dtype, scale=4)
        close(nfm.sym_matmul_solve(dj, dh, dg, dr), P.sym_solve(a, g, reg), dtype, scale=10)
        if k >= d:
            close(nfm.sym_matmul_solve(dj, dh, dg), P.sym_solve(a, g), dtype, scale=10)
        # diagonal Hessian (reference jhjn accepts it) and a scalar regulariser
        hd = h[..., :k].contiguous()
        if not (k == d and k <= 3):
            ad = P.full_to_sym(j.transpose(-1, -2) @ torch.diag_embed(hd) @ j)
            close(nfm.sym_matmul(dj, hd.to(DEV)), ad, dtype, scale=4)
            close(nfm.sym_matmul_solve(dj, hd.to(DEV), dg, 0.5), P.sym_solve(ad, g, 0.5), dtype, scale=10)
    # broadcasting: one Jacobian for the whole field
    j1 = torch.eye(3, dtype=dtype) * 1.5
    h = G.spd_packed(batch, 3, dtype, seed=3)
    g = G.vectors(batch, 3, dtype, seed=9)
    close(nfm.sym_matmul_solve(j1.to(DEV), h.to(DEV), g.to(DEV)), P.sym_solve(P.sym_matmul(j1.expand(batch, 3, 3), h), g), dtype, scale=10)


def test_partially_broadcast_operands_are_not_materialised(nfm):
    """One Hessian field for a batch of gradient fields (and the other way round): the leading
    batch dims are looped over with one launch each, on views -- no operand is copied."""
    from nitorch_fastmath_b200 import _lib
    dtype, n = torch.float32, 3
    b, x, y = 3, 40, 50
    mat1 = G.spd_packed((1, x, y), n, dtype, seed=1)           # (1, X, Y, 6): shared by the batch
    vec = G.vectors((b, x, y), n, dtype, seed=2)               # (B, X, Y, 3)
    want = P.sym_solve(mat1.expand(b, x, y, -1).contiguous(), vec)
    before = _lib.launch_count()
    got = nfm.sym_solve(mat1.to(DEV), vec.to(DEV))
    assert _lib.launch_count() - before == b                   # one launch per outer index, each on the TMA path
    assert _lib.load().nfm_last_path_was_tma() == 1
    close(got, want, dtype)
    close(nfm.sym_matvec(mat1.to(DEV), vec.to(DEV)), P.sym_matvec(mat1.expand(b, x, y, -1).contiguous(), vec), dtype)
    # per-image matrices, one vector field: (B, 1, 1, 6) with (1, X, Y, 3); and a regulariser field (1, X, Y, 3)
    matb = G.spd_packed((b, 1, 1), n, dtype, seed=3)
    vec1 = G.vectors((1, x, y), n, dtype, seed=4)
    reg1 = G.vectors((1, x, y), n, dtype, seed=5).abs()
    want = P.sym_solve(matb.expand(b, x, y, -1).contiguous(), vec1.expand(b, x, y, -1).contiguous(),
                       reg1.expand(b, x, y, -1).contiguous())
    out = torch.empty(b, x, y, n, device=DEV, dtype=dtype)
    assert nfm.sym_solve(matb.to(DEV), vec1.to(DEV), reg1.to(DEV), out=out) is out
    close(out, want, dtype)


@pytest.mark.parametrize("n", [3, 6])
def test_storage_offset_views_take_the_tma_path(nfm, n):
    """A dense view that starts one record into its storage is not 16-byte aligned; the first
    h < 4 matrices are peeled off (strided kernel) so that the rest is, and goes by TMA."""
    from nitorch_fastmath_b200 import _lib
    dtype, batch = torch.float32, 200_001
    mat = G.spd_packed(batch + 1, n, dtype, seed=n).to(DEV)
    vec = G.vectors(batch + 1, n, dtype, seed=n + 1).to(DEV)
    assert mat[1:].data_ptr() % 16 != 0 or vec[1:].data_ptr() % 16 != 0
    before = _lib.launch_count()
    x = nfm.sym_solve(mat[1:], vec[1:])
    assert _lib.load().nfm_last_path_was_tma() == 1
    assert _lib.launch_count() - before <= 3          # head, tiles (+ the < 4-matrix tail)
    close(x, P.sym_solve(mat[1:].cpu(), vec[1:].cpu()), dtype)
    assert torch.equal(x, nfm.sym_solve(mat[1:].clone(), vec[1:].clone()))
    inv = nfm.sym_invert(mat[1:])
    close(inv, P.sym_invert(mat[1:].cpu()), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [1, 3, 6, 10])
def test_many_right_hand_sides_and_right_division(nfm, dtype, n):
    """lmdiv with more than 4 right-hand sides and rmdiv run on the register-factorisation
    kernel (order templated, run-time loop over the right-hand sides); rmdiv solves
    b^T x_r = a_r natively -- no transposed copies."""
    batch = 5003
    a = _row_permuted(G.dense_shifted(batch, n, dtype, seed=n), seed=n)          # half of the lanes pivot
    spd = G.dense_spd(batch, n, dtype, seed=n + 1)
    from nitorch_fastmath_b200 import _lib
    lib = _lib.load()
    esize = 4 if dtype == torch.float32 else 8

    def staged(k):      # three warps' double buffers (+ transposition scratch) fit the 227 KB of shared memory
        def degree(length):
            words, g = length * esize // 4, 1
            while g < 32 and words % (2 * g) == 0:
                g *= 2
            return g // (esize // 4)
        buf = (32 * (n * n + n * k) * esize + 127) // 128 * 128
        ta, tb = degree(n * n) >= 16, degree(n * k) >= 16 and k < 4      # matrices / right-hand sides re-laid out
        scratch = (n * k if (tb and k > n) or not ta else n * n) * 33 * esize if ta or tb else 0
        return (232448 - 256) // (2 * (buf + 8) + scratch) >= 3

    for k in (5, 7, 12):
        b = G.vectors((batch, n), k, dtype, seed=k)
        close(nfm.lmdiv(a.to(DEV), b.to(DEV)), P.lmdiv(a, b), dtype, 2, scale=4)
        # dense aligned operands take the TMA-staged kernel whenever three warps' double buffers fit
        assert lib.nfm_last_path_was_tma() == (4 if staged(k) else 0)
        # ... which computes what the one-thread-per-system kernel computes, bit for bit (a view that is
        # not 16-byte aligned takes that kernel)
        if n > 1:
            pad_a = torch.empty(batch * n * n + 1, device=DEV, dtype=dtype)[1:].view(batch, n, n).copy_(a)
            assert pad_a.data_ptr() % 16 != 0
            ref = nfm.lmdiv(pad_a, b.to(DEV))
            assert lib.nfm_last_path_was_tma() == 0
            assert torch.equal(ref, nfm.lmdiv(a.to(DEV), b.to(DEV)))
        close(nfm.lmdiv(spd.to(DEV), b.to(DEV), "chol"), P.lmdiv(spd, b, "chol"), dtype, 2, scale=4)
    for k in (1, 3, 4, 9):
        r = G.vectors((batch, k), n, dtype, seed=20 + k)                          # (batch, k, n)
        want = (r.double() @ torch.linalg.inv(a.double())).to(dtype)              # the documented a @ inv(b)
        got = nfm.rmdiv(r.to(DEV), a.to(DEV))
        # 2..4 rows: the register kernels of lmdiv on the TMA tile / pool path, records read in the other
        # index order; 1 row and more than 4: the staged many-right-hand-sides kernel
        assert lib.nfm_last_path_was_tma() == ((3 if n >= 8 or (n >= 6 and esize == 8) else 1) if 2 <= k <= 4 else 4 if staged(k) else 0)
        close(got, want, dtype, 2, scale=4)
        want_c = (r.double() @ torch.linalg.inv(spd.double())).to(dtype)
        close(nfm.rmdiv(r.to(DEV), spd.to(DEV), "chol"), want_c, dtype, 2, scale=4)
        out = torch.empty(batch, k, n, device=DEV, dtype=dtype)
        assert nfm.rmdiv(r.to(DEV), a.to(DEV), out=out) is out and torch.equal(out, got)
    # the solutions may overwrite the right-hand sides (register kernels and the staged kernel alike)
    for k in (3, 6):
        b = G.vectors((batch, n), k, dtype, seed=90 + k).to(DEV)
        want = nfm.lmdiv(a.to(DEV), b)
        assert nfm.lmdiv(a.to(DEV), b, out=b) is b and torch.equal(b, want)
        r = G.vectors((batch, k), n, dtype, seed=95 + k).to(DEV)
        want = nfm.rmdiv(r, a.to(DEV))
        assert nfm.rmdiv(r, a.to(DEV), out=r) is r and torch.equal(r, want)
    # broadcasting: one system for the whole batch
    r = G.vectors((batch, 2), n, dtype, seed=77)
    close(nfm.rmdiv(r.to(DEV), a[0].to(DEV)), (r.double() @ torch.linalg.inv(a[0].double())).to(dtype), dtype, 2, scale=4)
