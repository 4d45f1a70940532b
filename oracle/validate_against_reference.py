"""Pin the oracle: compare oracle/ref_port.py with the real reference.

Against the unmodified reference (see oracle/load_reference.py):

    NFM_REFERENCE_ROOT=<nitorch-fastmath checkout> python -m oracle.validate_against_reference

For every routine on the hot path it feeds identical seeded inputs to the
reference (imported through oracle/load_reference.py) and to the restatement
and reports the worst absolute difference.  The closed forms (N <= 4, dense
n <= 3) and the LAPACK-backed branches are expected to agree BIT FOR BIT,
because the restatement keeps the reference's operation order.  Exit code is
non-zero on any mismatch.

``run(stored=...)`` makes the same checks against stored reference outputs
instead of calling the reference (tests/golden/oracle_pin_*.npz, written by
``run(record=...)`` from tests/golden/make_golden.py), so that
tests/test_oracle.py makes every check in every checkout.  To keep the files
small, exact checks store a fixed sample of PIN_ELEMS output elements and the
output's shape; checks to rounding store the whole output.
"""
from __future__ import annotations

import sys
import zlib

import numpy as np
import torch

from . import generators as G
from . import load_reference, ref_port as P


def _maxdiff(a, b):
    if a.shape != b.shape:
        return float("inf")
    if a.numel() == 0:
        return 0.0
    return float((a.double() - b.double()).abs().max())


PIN_ELEMS = 32   # elements stored per exactly compared output (the files stay small)
PIN_INPUT_ELEMS = 8


def _pick(name: str, t: torch.Tensor, count) -> torch.Tensor:
    """A fixed sample (seeded by ``name``) of ``count`` of the flattened elements of ``t``, in
    storage order; all of them when ``count`` is None or there are not more."""
    flat = t.contiguous().reshape(-1)
    if count is None or flat.numel() <= count:
        return flat
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    return flat[torch.randperm(flat.numel(), generator=g)[:count].sort().values]


def save_pin(path: str, record: dict) -> None:
    """Write a ``record`` of ``run`` (name -> 1-D array) as one .npz of a few packed arrays."""
    keys = sorted(record)
    packed = {"keys": np.array(keys), "dtypes": np.array([record[k].dtype.name for k in keys])}
    for dt in sorted(set(packed["dtypes"])):
        part = [record[k] for k in keys if record[k].dtype.name == dt]
        packed["values_" + dt] = np.concatenate(part)
        packed["bounds_" + dt] = np.cumsum([0] + [a.size for a in part])
    np.savez_compressed(path, **packed)


def load_pin(*paths: str) -> dict:
    """The mapping ``save_pin`` wrote, merged over ``paths``."""
    out = {}
    for path in paths:
        z = np.load(path)
        seen = {}
        for key, dt in zip(z["keys"].tolist(), z["dtypes"].tolist()):
            i = seen[dt] = seen.get(dt, -1) + 1
            b = z["bounds_" + dt]
            out[key] = z["values_" + dt][b[i]:b[i + 1]]
    return out


def run(verbose: bool = True, stored=None, record=None) -> int:
    """Number of mismatches.

    ``record``: a dict that receives, per check, the shape of the reference output (``shape
    <name>``) and its elements (``out <name>``: all of them for checks to rounding, a fixed
    sample of PIN_ELEMS for exact ones), and a fixed sample of PIN_INPUT_ELEMS elements of
    every generated input (``in <key>``).  ``stored``: such a mapping (``load_pin``); when
    given, the reference is not imported, the
    inputs are regenerated and must reproduce their stored samples, and the port is compared
    with the stored outputs at each check's own exactness."""
    if stored is None:
        ref_sym, ref_bat, ref_sugar = load_reference.load()
    bad = 0
    rows = []

    def data(key, make):
        t = make()
        sample = _pick(key, t, PIN_INPUT_ELEMS)
        if stored is not None and not torch.equal(sample, torch.from_numpy(stored["in " + key])):
            raise RuntimeError(f"oracle/generators.py no longer reproduces the stored input {key!r}")
        if record is not None:
            record["in " + key] = sample.numpy()
        return t

    def check(name, got, want, exact=True, rtol=0.0):
        """``want``: zero-argument call of the reference; ``rtol`` scales with max |want|."""
        nonlocal bad
        if stored is not None:
            if tuple(got.shape) != tuple(int(s) for s in stored["shape " + name]):
                rows.append((name, float("inf"), False))
                bad += 1
                return
            got, want = _pick(name, got, PIN_ELEMS if exact else None), torch.from_numpy(stored["out " + name])
        else:
            want = want()
            if record is not None:
                record["shape " + name] = np.array(want.shape, dtype=np.int64)
                record["out " + name] = _pick(name, want, PIN_ELEMS if exact else None).numpy()
        d = _maxdiff(got, want)
        ok = (d == 0.0) if exact else (d <= rtol * float(want.abs().max()))
        ok = ok and got.dtype == want.dtype
        rows.append((name, d, ok))
        if not ok:
            bad += 1

    for dtype in (torch.float32, torch.float64):
        tag = "f32" if dtype == torch.float32 else "f64"
        for n in range(1, 11):
            mat = data(f"mat n={n} {tag}", lambda: G.spd_packed((7, 33), n, dtype, seed=n))
            vec = data(f"vec n={n} {tag}", lambda: G.vectors((7, 33), n, dtype, seed=100 + n))
            inp = data(f"inp n={n} {tag}", lambda: G.vectors((7, 33), n, dtype, seed=200 + n))
            check(f"sym_matvec n={n} {tag}", P.sym_matvec(mat, vec), lambda: ref_sym.sym_matvec(mat, vec))
            check(f"sym_addmatvec n={n} {tag}", P.sym_addmatvec(inp, mat, vec),
                  lambda: inp + ref_sym.sym_matvec(mat, vec))
            check(f"sym_solve n={n} {tag}", P.sym_solve(mat, vec), lambda: ref_sym.sym_solve(mat, vec))
            check(f"sym_invert n={n} {tag}", P.sym_invert(mat), lambda: ref_sym.sym_invert(mat))
            check(f"sym_invert diag n={n} {tag}", P.sym_invert(mat, True), lambda: ref_sym.sym_invert(mat, True))
            check(f"sym_to_full n={n} {tag}", P.sym_to_full(mat), lambda: ref_sym.sym_to_full(mat))
            # documented regulariser semantics == reference on pre-shifted diagonal
            shifted = mat.clone()
            shifted[..., :n] += 0.25
            check(f"sym_solve diag=0.25 n={n} {tag}", P.sym_solve(mat, vec, 0.25),
                  lambda: ref_sym.sym_solve(shifted, vec))
            # broadcasting of either operand
            check(f"sym_solve bcast-vec n={n} {tag}", P.sym_solve(mat, vec[0, 0]),
                  lambda: ref_sym.sym_solve(mat, vec[0, 0]))
            check(f"sym_solve bcast-mat n={n} {tag}", P.sym_solve(mat[0, 0], vec),
                  lambda: ref_sym.sym_solve(mat[0, 0], vec))
        # eps exactly as written: only N == 2 runs in the reference
        mat = data(f"eps mat n=2 {tag}", lambda: G.spd_packed(50, 2, dtype, seed=5))
        vec = data(f"eps vec n=2 {tag}", lambda: G.vectors(50, 2, dtype, seed=6))
        check(f"sym_solve eps-as-written n=2 {tag}", P.sym_solve_ref_eps(mat, vec, 0.1),
              lambda: ref_sym.sym_solve(mat, vec, 0.1))
        # empty batch
        check(f"sym_solve empty {tag}", P.sym_solve(mat[:0], vec[:0]), lambda: ref_sym.sym_solve(mat[:0], vec[:0]))

        for n in range(1, 11):
            a = data(f"dense n={n} {tag}", lambda: G.dense_shifted((5, 21), n, dtype, seed=n))
            b = data(f"dense vec n={n} {tag}", lambda: G.vectors((5, 21), n, dtype, seed=50 + n))
            check(f"batchinv n={n} {tag}", P.batchinv(a), lambda: ref_bat.batchinv(a))
            check(f"batchdet n={n} {tag}", P.batchdet(a), lambda: ref_bat.batchdet(a))
            check(f"batchmatvec n={n} {tag}", P.batchmatvec(a, b), lambda: ref_bat.batchmatvec(a, b))
            check(f"solvevec lu n={n} {tag}", P.solvevec(a, b, "lu"), lambda: ref_sugar.solvevec(a, b, "lu"))
            check(f"inv lu n={n} {tag}", P.inv(a, "lu"), lambda: ref_sugar.inv(a, "lu"))
            s = data(f"dense spd n={n} {tag}", lambda: G.dense_spd((5, 21), n, dtype, seed=n))
            check(f"solvevec chol n={n} {tag}", P.solvevec(s, b, "chol"), lambda: ref_sugar.solvevec(s, b, "chol"))
            check(f"inv chol n={n} {tag}", P.inv(s, "chol"), lambda: ref_sugar.inv(s, "chol"))
            rhs = data(f"dense rhs n={n} {tag}", lambda: G.vectors((5, 21, n), 3, dtype, seed=70 + n))
            check(f"lmdiv lu k=3 n={n} {tag}", P.lmdiv(a, rhs, "lu"), lambda: ref_sugar.lmdiv(a, rhs, "lu"))
        # the closed forms the reference only dispatches to on CUDA, run on CPU
        for n in (2, 3):
            a = data(f"dense n={n} {tag}", lambda: G.dense_shifted((5, 21), n, dtype, seed=n))
            c = a.movedim(-1, 0).movedim(-1, 0)
            check(f"closed_inv n={n} {tag}", P.closed_inv(a),
                  lambda: (ref_bat.inv2 if n == 2 else ref_bat.inv3)(c).movedim(0, -1).movedim(0, -1))
            check(f"closed_det n={n} {tag}", P.closed_det(a), lambda: (ref_bat.det2 if n == 2 else ref_bat.det3)(c))

    # "next" rows: sym_outer bit for bit; sym_matmul restated as behaviour (dense
    # congruence incl. the J H J^T quirk of the unrolled k == d <= 3 branches): to rounding
    for dtype, tol in ((torch.float32, 2e-5), (torch.float64, 1e-13)):
        tag = "f32" if dtype == torch.float32 else "f64"
        x = data(f"outer x {tag}", lambda: G.vectors((4, 9), 5, dtype, seed=3))
        check(f"sym_outer {tag}", P.sym_outer(x), lambda: ref_sym.sym_outer(x))
        for k, d in ((1, 1), (2, 2), (3, 3), (4, 4), (2, 3), (4, 2), (5, 3)):
            jac = data(f"matmul j k={k} d={d} {tag}", lambda: G.vectors((4, 9, k), d, dtype, seed=10 * k + d))
            h = data(f"matmul h k={k} d={d} {tag}", lambda: G.spd_packed((4, 9), k, dtype, seed=k))
            check(f"sym_matmul k={k} d={d} {tag}", P.sym_matmul(jac, h), lambda: ref_sym.sym_matmul(jac, h),
                  exact=False, rtol=tol)
        # sym_det is not compared in general: the reference takes the order from a batch dimension
        # (_impl/sym.py:434), so it raises or is wrong unless the batch size happens to
        # equal N(N+1)/2 -- e.g. N = 3 with a batch of exactly 6:
        m3 = data(f"det mat n=3 {tag}", lambda: G.spd_packed(6, 3, dtype, seed=8))
        check(f"sym_det n=3 batch=6 {tag}", P.sym_det(m3), lambda: ref_sym.sym_det(m3), exact=False, rtol=tol)

    if verbose:
        for name, d, ok in rows:
            if not ok or d != 0.0:
                print(f"{'ok ' if ok else 'BAD'} {name:40s} maxdiff={d:.3e}")
        print(f"{len(rows)} checks, {bad} mismatches "
              f"({sum(1 for r in rows if r[1] == 0.0)} bit-exact)")
    return bad


if __name__ == "__main__":
    sys.exit(1 if run() else 0)
