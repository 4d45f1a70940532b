"""Every shape the Gauss-Newton builders accept, and every run-time-sized kernel past its grid cap.

``sym_matmul`` and its backward have register kernels for the shapes ``fused_shape_built``
names (k, d <= 6, and k <= 10 with d <= 3; mode 1, J H J^T, for k = d <= 3) and run the
run-time-sized ``matmul_rt_kernel`` / ``matmul_backward_rt_kernel`` for the other 52 of the
100 (k, d).  Here every shape is checked against a float64 reference on the GPU, in fp32 and
fp64: the forward with a packed, a diagonal and a broadcast operand, the backward for each
``which`` (dJ, dH, both), views against dense copies bit for bit, the ABI modes no Python
path selects, and ``sym_matmul_solve`` at each of its 48 shapes.

Register-kernel shapes run a ragged batch (full TMA tiles, a partial tile and a strided
tail).  The run-time-sized kernels (``nfm_generic.cu``) cap their grid at 16 blocks of 128
threads per SM and walk the rest with a grid-stride loop; they run a batch on which every
thread takes at least two steps of that loop.

The return codes of the entries with NULL operands pin which shapes each one accepts; they
run without a GPU.
"""
from __future__ import annotations

import pytest
import torch

from conftest import TOL
from nitorch_fastmath_b200 import _lib
from oracle import ref_port as P

DEV = "cuda:0"
NS = range(1, _lib.MAX_N + 1)
SHAPES = [(k, d) for k in NS for d in NS]
DTYPES = [torch.float32, torch.float64]
RAGGED = 20_011          # full TMA tiles, a partial tile and a strided tail
VIEWS = 4099             # batch of the view checks (head peel: more than 64 matrices)
SCALE = 10               # products of three matrices (a solve for sym_matmul_solve) at the per-matrix bars
E_UNSUPPORTED, E_BADARG = -1, -2


def built(k, d):
    """``fused_shape_built`` of csrc/nfm_impl.cuh: the shapes with register kernels."""
    return 1 <= k <= _lib.MAX_N and 1 <= d <= _lib.MAX_N and ((k <= 6 and d <= 6) or d <= 3)


def mode_of(k, d):
    return 1 if (k == d and k <= 3) else 0


def past_grid_cap(per_matrix):
    """A batch on which a run-time-sized kernel with ``per_matrix`` threads of work per matrix
    runs its grid-stride loop at least twice (grid: at most 16 x SMs blocks of 128 threads),
    with a ragged remainder."""
    threads = 16 * torch.cuda.get_device_properties(0).multi_processor_count * 128
    return -(-(2 * threads + 1237) // per_matrix)


def _dtype_code(dtype):
    return _lib.F32 if dtype == torch.float32 else _lib.F64


# ---------------------------------------------------------------------------
# CPU: the shapes each entry accepts
# ---------------------------------------------------------------------------

def test_sym_matmul_solve_accepts_exactly_the_built_shapes_without_a_gpu():
    lib = _lib.load()
    for dt in (_lib.F32, _lib.F64):
        for k in range(0, _lib.MAX_N + 2):
            for d in range(0, _lib.MAX_N + 2):
                for mode in (0, 1, 2):
                    ok = built(k, d) and (mode == 0 or (mode == 1 and k == d and k <= 3))
                    rc = lib.nfm_sym_matmul_solve(dt, k, d, mode, 4, None, 0, None, 0, None, 0, None, 0, None, 0, None)
                    assert rc == (E_BADARG if ok else E_UNSUPPORTED), (dt, k, d, mode, rc)


def test_sym_matmul_and_its_backward_accept_every_shape_without_a_gpu():
    lib = _lib.load()
    for dt in (_lib.F32, _lib.F64):
        for k in range(0, _lib.MAX_N + 2):
            for d in range(0, _lib.MAX_N + 2):
                for mode in (0, 1, 2):
                    ok = 1 <= k <= _lib.MAX_N and 1 <= d <= _lib.MAX_N and (mode == 0 or (mode == 1 and k == d))
                    rc = lib.nfm_sym_matmul(dt, k, d, mode, 4, None, 0, None, 0, None, 0, None)
                    assert rc == (E_BADARG if ok else E_UNSUPPORTED), (dt, k, d, mode, rc)
                    for which in (0, 1, 2, 3, 4):
                        rc = lib.nfm_sym_matmul_backward(dt, k, d, mode, which, 4, None, 0, None, 0, None, 0, None, 0, None)
                        want = E_BADARG if ok and 1 <= which <= 3 else E_UNSUPPORTED
                        assert rc == want, (dt, k, d, mode, which, rc)


# ---------------------------------------------------------------------------
# inputs and float64 references, on the GPU
# ---------------------------------------------------------------------------

def _randn(shape, seed, dtype=torch.float64):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, device=DEV, dtype=torch.float64, generator=g).to(dtype)


def _jac(b, k, d, dtype, seed):
    """0.1 randn plus ones on the leading diagonal: J^T H J (+ diag d) stays well conditioned."""
    return (0.1 * _randn((b, k, d), seed) + torch.eye(k, d, device=DEV, dtype=torch.float64)).to(dtype)


def _pidx(n):
    idx = torch.empty(n, n, dtype=torch.long)
    for i in range(n):
        for j in range(n):
            idx[i, j] = P.packed_index(n, i, j)
    return idx.to(DEV)


def _unpack(p, n):
    return p.double()[..., _pidx(n)]


def _pack(m, double_off=False):
    n = m.shape[-1]
    iu = torch.triu_indices(n, n, 1, device=DEV)
    off = m[..., iu[0], iu[1]]
    return torch.cat([m.diagonal(0, -1, -2), 2 * off if double_off else off], -1)


def _spd(b, n, dtype, seed):
    a = _randn((b, n, n), seed)
    full = a @ a.transpose(-1, -2)
    full.diagonal(0, -1, -2).add_(n)
    return _pack(full).to(dtype)


def _ghat(g, n):
    f = _unpack(g, n)
    return (f + torch.diag_embed(f.diagonal(0, -1, -2))) / 2


def _jhj(j, hf, mode):
    """Y = J^T H J (mode 0) or J H J^T (mode 1), full, float64."""
    j = j.double()
    return j @ hf @ j.transpose(-1, -2) if mode == 1 else j.transpose(-1, -2) @ hf @ j


def _matmul_grads(j, h, g, k, d, mode):
    """dJ = 2 H J G^, dH = pack(J G^ J^T) (mode 1: dJ = 2 G^ J H, dH = pack(J^T G^ J)), float64."""
    j = j.double()
    kh, ko = (d, k) if mode == 1 else (k, d)
    hf, gh = _unpack(h, kh), _ghat(g, ko)
    if mode == 1:
        return 2 * gh @ j @ hf, _pack(j.transpose(-1, -2) @ gh @ j, True)
    return 2 * hf @ j @ gh, _pack(j @ gh @ j.transpose(-1, -2), True)


def _err(got, want, rec, den=None):
    """Worst per-matrix norm-wise relative error over the trailing ``rec`` dims, relative to ``den`` if given."""
    dims = tuple(range(-rec, 0))
    num = (got.double() - want).pow(2).sum(dims).sqrt()
    den = want if den is None else den
    return float((num / den.pow(2).sum(dims).sqrt().clamp_min(1e-300)).max())


def _check(got, want, dtype, rec=1, what="", den=None):
    """``den``: for sums of products of random signs, the same formula on the magnitudes of the inputs
    (a record whose entries all nearly cancel has no exact digits to compare)."""
    assert got.dtype == dtype and got.shape == want.shape, (what, got.dtype, got.shape, want.shape)
    err = _err(got, want, rec, den)
    assert err <= TOL[dtype] * SCALE, f"{what}: worst rel err {err:.3e}"


_PRIME = {}


def _prime():
    """A call on the TMA tile kernel, so that the next launch record is that call's own."""
    nfm = _nfm()
    if "x" not in _PRIME:
        _PRIME["x"] = _randn((VIEWS, 3), 99, torch.float32)
    nfm.sym_outer(_PRIME["x"])
    assert _path() == 1 and _kind() == 1


def _nfm():
    import nitorch_fastmath_b200 as pkg
    return pkg


def _path():
    return int(_lib.load().nfm_last_path_was_tma())


def _kind():
    return _lib.last_launch_shape()["kind"]


def _assert_path(k, d, what):
    """Register kernels on the TMA tile kernel, the other shapes on the run-time-sized kernel."""
    if built(k, d):
        assert _path() == 1, (what, k, d, _path())
    else:
        assert _path() == 0 and _kind() == 0, (what, k, d, _path(), _lib.last_launch_shape())


# ---------------------------------------------------------------------------
# sym_matmul forward: all 100 shapes
# ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("k,d", SHAPES)
def test_sym_matmul_every_shape(k, d, dtype):
    nfm = _nfm()
    mode = mode_of(k, d)
    kh = d if mode == 1 else k
    b = RAGGED if built(k, d) else past_grid_cap(1)
    j, h = _jac(b, k, d, dtype, 1), _spd(b, kh, dtype, 2)
    hf = _unpack(h, kh)
    _prime()
    y = nfm.sym_matmul(j, h)
    _assert_path(k, d, "sym_matmul")
    _check(y, _pack(_jhj(j, hf, mode)), dtype, what=f"packed h {k}x{d}")
    del y
    hd = (_randn((b, kh), 3).abs() + 0.1).to(dtype)
    _check(nfm.sym_matmul(j, hd), _pack(_jhj(j, torch.diag_embed(hd.double()), mode)), dtype, what=f"diagonal h {k}x{d}")
    del hd
    _check(nfm.sym_matmul(j[0], h), _pack(_jhj(j[0].expand(b, k, d), hf, mode)), dtype, what=f"one J {k}x{d}")
    _check(nfm.sym_matmul(j, h[0]), _pack(_jhj(j, hf[0].expand(b, kh, kh), mode)), dtype, what=f"one H {k}x{d}")
    # a head-peeled view (not 16-byte aligned) and every other matrix: the bits of the dense call on copies
    jv, hv = j[:VIEWS + 1], h[:VIEWS + 1]
    for sl in (slice(1, None), slice(None, None, 2)):
        assert torch.equal(nfm.sym_matmul(jv[sl], hv[sl]), nfm.sym_matmul(jv[sl].contiguous(), hv[sl].contiguous())), (k, d, sl)


# ---------------------------------------------------------------------------
# sym_matmul backward: all 100 shapes, dJ / dH / both
# ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("k,d", SHAPES)
def test_matmul_backward_every_shape(k, d, dtype):
    from nitorch_fastmath_b200 import _autograd as A
    mode = mode_of(k, d)
    kh, ko = (d, k) if mode == 1 else (k, d)
    b = RAGGED if built(k, d) else past_grid_cap(1)
    j, h, g = _jac(b, k, d, dtype, 1), _spd(b, kh, dtype, 2), _randn((b, ko * (ko + 1) // 2), 3, dtype)
    want_j, want_h = _matmul_grads(j, h, g, k, d, mode)
    mag_j, mag_h = _matmul_grads(j.abs(), h.abs(), g.abs(), k, d, mode)
    got = {}
    for which in (1, 2, 3):
        _prime()
        got[which] = A.matmul_backward(j, h, g, which)
        _assert_path(k, d, f"matmul_backward which={which}")
    assert got[1][1] is None and got[2][0] is None
    _check(got[1][0], want_j, dtype, 2, f"dJ {k}x{d} which=1", mag_j)
    _check(got[2][1], want_h, dtype, 1, f"dH {k}x{d} which=2", mag_h)
    _check(got[3][0], want_j, dtype, 2, f"dJ {k}x{d} which=3", mag_j)
    _check(got[3][1], want_h, dtype, 1, f"dH {k}x{d} which=3", mag_h)
    # (different instantiations: equal within the bar, not bit for bit)
    _check(got[3][0], got[1][0].double(), dtype, 2, f"dJ {k}x{d} which=3 against which=1", mag_j)
    _check(got[3][1], got[2][1].double(), dtype, 1, f"dH {k}x{d} which=3 against which=2", mag_h)
    del got, want_j, want_h, mag_j, mag_h
    jv, hv, gv = j[:VIEWS + 1], h[:VIEWS + 1], g[:VIEWS + 1]
    for which in (1, 2, 3):
        for sl in (slice(1, None), slice(None, None, 2)):
            view = A.matmul_backward(jv[sl], hv[sl], gv[sl], which)
            dense = A.matmul_backward(jv[sl].contiguous(), hv[sl].contiguous(), gv[sl].contiguous(), which)
            for a, c in zip(view, dense):
                assert (a is None and c is None) or torch.equal(a, c), (k, d, which, sl)


# ---------------------------------------------------------------------------
# the ABI modes no Python path selects
# ---------------------------------------------------------------------------

ABI_MODES = [(0, n) for n in (1, 2, 3)] + [(1, n) for n in range(4, _lib.MAX_N + 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("mode,n", ABI_MODES)
def test_abi_only_modes(mode, n, dtype):
    """J^T H J at k = d <= 3 (register kernels) and J H J^T at k = d >= 4 (run-time-sized kernels),
    forward and backward, through the C ABI."""
    lib = _lib.load()
    nn = n * (n + 1) // 2
    tile = mode == 0     # mode 0 at n <= 3 is built; mode 1 above 3 runs on the run-time-sized kernels
    b = RAGGED if tile else past_grid_cap(1)
    j, h, g = _jac(b, n, n, dtype, 1), _spd(b, n, dtype, 2), _randn((b, nn), 3, dtype)
    stream = torch.cuda.current_stream().cuda_stream
    dt = _dtype_code(dtype)

    def expect_path():
        if tile:
            assert _path() == 1, (mode, n)
        else:
            assert _path() == 0 and _kind() == 0, (mode, n, _lib.last_launch_shape())

    y = torch.empty(b, nn, device=DEV, dtype=dtype)
    _prime()
    _lib.check(lib.nfm_sym_matmul(dt, n, n, mode, b, j.data_ptr(), n * n, h.data_ptr(), nn, y.data_ptr(), nn, stream),
               "nfm_sym_matmul")
    expect_path()
    _check(y, _pack(_jhj(j, _unpack(h, n), mode)), dtype, what=f"forward mode {mode} n={n}")
    del y
    want_j, want_h = _matmul_grads(j, h, g, n, n, mode)
    mag_j, mag_h = _matmul_grads(j.abs(), h.abs(), g.abs(), n, n, mode)
    for which in (1, 2, 3):
        rec = (n * n if which & 1 else 0) + (nn if which & 2 else 0)
        out = torch.empty(b, rec, device=DEV, dtype=dtype)
        _prime()
        _lib.check(lib.nfm_sym_matmul_backward(dt, n, n, mode, which, b, j.data_ptr(), n * n, h.data_ptr(), nn,
                                               g.data_ptr(), nn, out.data_ptr(), rec, stream), "nfm_sym_matmul_backward")
        expect_path()
        if which & 1:
            _check(out[:, :n * n].unflatten(-1, (n, n)), want_j, dtype, 2, f"dJ mode {mode} n={n} which={which}", mag_j)
        if which & 2:
            _check(out[:, rec - nn:], want_h, dtype, 1, f"dH mode {mode} n={n} which={which}", mag_h)
        del out


# ---------------------------------------------------------------------------
# sym_matmul_solve: its 48 shapes
# ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("k,d", [s for s in SHAPES if built(*s)])
def test_sym_matmul_solve_every_built_shape(k, d, dtype):
    nfm = _nfm()
    mode = mode_of(k, d)
    kh = d if mode == 1 else k
    b = RAGGED
    j, h, g = _jac(b, k, d, dtype, 1), _spd(b, kh, dtype, 2), _randn((b, d), 3, dtype)
    a = _jhj(j, _unpack(h, kh), mode)
    reg_t = (1 + _randn((b, d), 4).abs()).to(dtype)
    regs = [("tensor", reg_t, torch.diag_embed(reg_t.double())),
            ("float", 1.0, torch.eye(d, device=DEV, dtype=torch.float64))]
    if k >= d:   # J^T H J has full rank
        regs.append(("none", None, 0))
    for name, reg, shift in regs:
        x = nfm.sym_matmul_solve(j, h, g, reg)
        assert _path() == 1, (k, d, name)
        want = torch.linalg.solve(a + shift, g.double()[..., None])[..., 0]
        _check(x, want, dtype, what=f"{k}x{d} regulariser {name}")


@pytest.mark.gpu
def test_sym_matmul_solve_rejects_the_other_shapes():
    nfm = _nfm()
    for k, d in SHAPES:
        if built(k, d):
            continue
        j, h, g = torch.ones(4, k, d, device=DEV), torch.ones(4, k * (k + 1) // 2, device=DEV), torch.ones(4, d, device=DEV)
        with pytest.raises(ValueError):
            nfm.sym_matmul_solve(j, h, g, 1.0)


# ---------------------------------------------------------------------------
# the launch record after a run-time-sized kernel
# ---------------------------------------------------------------------------

@pytest.mark.gpu
def test_run_time_sized_entries_reset_the_launch_record():
    """After a TMA launch, sym_matmul on an unbuilt shape and a rectangular batchmatvec report
    the strided path and no bulk launch, not the previous call's record."""
    nfm = _nfm()
    j, h = _jac(VIEWS, 8, 5, torch.float32, 1), _spd(VIEWS, 8, torch.float32, 2)
    a, v = _randn((VIEWS, 3, 5), 3, torch.float32), _randn((VIEWS, 5), 4, torch.float32)
    for call in (lambda: nfm.sym_matmul(j, h), lambda: nfm.batchmatvec(a, v)):
        _prime()
        call()
        assert _path() == 0 and _lib.last_launch_shape()["kind"] == 0, _lib.last_launch_shape()


# ---------------------------------------------------------------------------
# run-time-sized dense kernels past the grid cap
# ---------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_run_time_sized_dense_kernels_past_the_grid_cap(dtype):
    """outer_rt_kernel (one thread per element): the lmdiv gradient with 8 right-hand sides and the
    rectangular batchmatvec gradient; matvec_rt_kernel (one thread per output row): the rectangular
    batchmatvec and its transposed form."""
    from nitorch_fastmath_b200 import _autograd as A
    nfm = _nfm()
    n, kk = 4, 8
    b = past_grid_cap(n * n)
    for rows, sym, sign in ((False, False, -1), (True, True, 1)):
        u = _randn((b, kk, n) if rows else (b, n, kk), 1, dtype)
        w = _randn((b, kk, n) if rows else (b, n, kk), 2, dtype)
        got = A.dense_outer(u, w, rows, sym, sign)
        assert _path() == 0 and _kind() == 0
        u, w = u.double(), w.double()
        m = u.transpose(-1, -2) @ w if rows else u @ w.transpose(-1, -2)
        mag = u.abs().transpose(-1, -2) @ w.abs() if rows else u.abs() @ w.abs().transpose(-1, -2)
        _check(got, sign * ((m + m.transpose(-1, -2)) / 2 if sym else m), dtype, 2, f"outer k={kk} rows={rows}", mag)
        del u, w, got, m, mag
    m, n = 3, 5
    b = past_grid_cap(m)
    gv, v = _randn((b, m), 3, dtype), _randn((b, n), 4, dtype)
    _check(A.dense_outer(gv[..., None], v[..., None], False, False, 1), gv.double()[..., None] * v.double()[..., None, :],
           dtype, 2, "outer 3x5")
    assert _path() == 0 and _kind() == 0
    a = _randn((b, m, n), 5, dtype)
    _prime()
    _check(nfm.batchmatvec(a, v), (a.double() @ v.double()[..., None])[..., 0], dtype, 1, "batchmatvec 3x5",
           (a.double().abs() @ v.double().abs()[..., None])[..., 0])
    assert _path() == 0 and _kind() == 0
    _check(A.dense_tmatvec(a, gv), (a.double().transpose(-1, -2) @ gv.double()[..., None])[..., 0], dtype, 1, "tmatvec 3x5",
           (a.double().abs().transpose(-1, -2) @ gv.double().abs()[..., None])[..., 0])
    assert _path() == 0 and _kind() == 0
