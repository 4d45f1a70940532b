"""The oracle (oracle/ref_port.py) against the fixtures the REAL reference
produced (tests/golden/make_golden.py), bit for bit against the stored outputs
of oracle/validate_against_reference.py, and -- when the unmodified reference
is installed (oracle/load_reference.py: NFM_REFERENCE_ROOT or baseline/_ref) --
against the reference itself.  CPU only."""
import os

import pytest
import torch

from conftest import GOLDEN, TAGS
from oracle import generators as G
from oracle import load_reference
from oracle import ref_port as P

DTYPES = [torch.float32, torch.float64]
# fixtures were produced by LAPACK / vectorised torch kernels of one build;
# another CPU may round the last bit differently
FIX_TOL = {torch.float32: 2e-6, torch.float64: 5e-15}


def _close(a, b, dtype, rec=1):
    assert a.shape == b.shape and a.dtype == b.dtype
    assert G.rel_err(a, b, rec) <= FIX_TOL[dtype]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_sym_against_golden(sym_golden, dtype, n):
    k = f"{TAGS[dtype]}_n{n}"
    mat, vec, inp, reg = (sym_golden(f"{k}_{s}") for s in ("mat", "vec", "inp", "reg"))
    _close(P.sym_matvec(mat, vec), sym_golden(f"{k}_matvec"), dtype)
    _close(P.sym_addmatvec(inp, mat, vec), sym_golden(f"{k}_addmatvec"), dtype)
    _close(P.sym_submatvec(inp, mat, vec), sym_golden(f"{k}_submatvec"), dtype)
    _close(P.sym_solve(mat, vec), sym_golden(f"{k}_solve"), dtype)
    _close(P.sym_solve(mat, vec, reg), sym_golden(f"{k}_solve_reg"), dtype)
    _close(P.sym_invert(mat), sym_golden(f"{k}_invert"), dtype)
    _close(P.sym_invert(mat, True), sym_golden(f"{k}_invert_diag"), dtype)
    _close(P.sym_to_full(mat), sym_golden(f"{k}_full"), dtype, 2)
    _close(P.sym_solve(sym_golden(f"{k}_ind_mat"), vec), sym_golden(f"{k}_ind_solve"), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_eps_as_written(sym_golden, dtype):
    t = TAGS[dtype]
    got = P.sym_solve_ref_eps(sym_golden(f"{t}_eps2_mat"), sym_golden(f"{t}_eps2_vec"), 0.1)
    _close(got, sym_golden(f"{t}_eps2_solve"), dtype)
    # as written the reference adds eps[0] to BOTH diagonal entries for N == 2,
    # which coincides with the documented semantics for a scalar eps
    _close(P.sym_solve(sym_golden(f"{t}_eps2_mat"), sym_golden(f"{t}_eps2_vec"), 0.1),
           sym_golden(f"{t}_eps2_solve"), dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", range(1, 11))
def test_dense_against_golden(dense_golden, dtype, n):
    k = f"{TAGS[dtype]}_n{n}"
    a, b, s, rhs = (dense_golden(f"{k}_{x}") for x in ("a", "b", "spd", "rhs"))
    _close(P.batchinv(a), dense_golden(f"{k}_inv"), dtype, 2)
    _close(P.batchdet(a), dense_golden(f"{k}_det"), dtype, 0)
    _close(P.batchmatvec(a, b), dense_golden(f"{k}_matvec"), dtype)
    _close(P.solvevec(a, b, "lu"), dense_golden(f"{k}_solve_lu"), dtype)
    _close(P.solvevec(s, b, "chol"), dense_golden(f"{k}_solve_chol"), dtype)
    _close(P.lmdiv(a, rhs, "lu"), dense_golden(f"{k}_lmdiv_lu"), dtype, 2)
    _close(P.inv(s, "chol"), dense_golden(f"{k}_inv_chol"), dtype, 2)
    if n in (2, 3):
        _close(P.closed_inv(a), dense_golden(f"{k}_closed_inv"), dtype, 2)
        _close(P.closed_det(a), dense_golden(f"{k}_closed_det"), dtype, 0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_next_rows_against_golden(extra_golden, dtype):
    t = TAGS[dtype]
    for n in (1, 2, 3, 5, 10):
        _close(P.sym_outer(extra_golden(f"{t}_outer{n}_x")), extra_golden(f"{t}_outer{n}"), dtype)
    for k, d in ((1, 1), (2, 2), (3, 3), (4, 4), (2, 3), (4, 2), (3, 1), (5, 3), (6, 6)):
        got = P.sym_matmul(extra_golden(f"{t}_jhj{k}x{d}_j"), extra_golden(f"{t}_jhj{k}x{d}_h"))
        assert G.rel_err(got, extra_golden(f"{t}_jhj{k}x{d}")) <= (2e-6 if dtype == torch.float32 else 1e-14)


def test_known_answers():
    """Analytic KATs (the reference ships none, SURVEY.md section 8c)."""
    # [[2,1],[1,2]] packed = [2,2,1]; inverse = 1/3 [[2,-1],[-1,2]]
    m = torch.tensor([2.0, 2.0, 1.0], dtype=torch.float64)
    assert torch.allclose(P.sym_invert(m), torch.tensor([2 / 3, 2 / 3, -1 / 3], dtype=torch.float64))
    assert torch.allclose(P.sym_solve(m, torch.tensor([3.0, 0.0], dtype=torch.float64)),
                          torch.tensor([2.0, -1.0], dtype=torch.float64))
    # identity of every order
    for n in range(1, 11):
        eye = torch.cat([torch.ones(n), torch.zeros(n * (n - 1) // 2)]).double()
        v = torch.arange(1.0, n + 1).double()
        assert torch.equal(P.sym_matvec(eye[None], v[None])[0], v)
        assert torch.allclose(P.sym_solve(eye, v), v)
        assert torch.allclose(P.sym_invert(eye), eye)
    # packed order: N=3 -> [a00 a11 a22 a01 a02 a12]
    full = P.sym_to_full(torch.arange(6.0))
    assert full.tolist() == [[0, 3, 4], [3, 1, 5], [4, 5, 2]]
    assert [P.packed_index(4, i, j) for i, j in P.packed_order(4)] == list(range(10))


def test_singular_closed_forms_do_not_raise():
    m = torch.zeros(4, 6)
    x = P.sym_solve(m, torch.ones(4, 3))
    assert not torch.isfinite(x).any()


def test_oracle_is_bit_identical_to_reference():
    """The 370 checks of oracle/validate_against_reference.py, each at its own exactness,
    against the reference outputs stored in tests/golden/oracle_pin_*.npz -- and against
    the reference itself where it is installed."""
    from oracle import validate_against_reference as V
    stored = V.load_pin(*(os.path.join(GOLDEN, f"oracle_pin_{t}.npz") for t in ("f32", "f64")))
    assert V.run(verbose=False, stored=stored) == 0
    if load_reference.available():
        assert V.run(verbose=False) == 0
