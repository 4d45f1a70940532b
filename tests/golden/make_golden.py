"""Generate the golden fixtures from the REAL reference.

    NFM_REFERENCE_ROOT=<nitorch-fastmath checkout> python tests/golden/make_golden.py

Imports the reference through oracle/load_reference.py, feeds it seeded
inputs and stores inputs + reference outputs in ``tests/golden/*.npz``.  The
reference itself holds no golden vectors for this path (SURVEY.md section 8c)
and is not part of this repository, so these files are the stored pin:
tests/test_oracle.py checks the oracle against them on CPU and
tests/test_gpu_parity.py checks the CUDA path against them on the B200.

``oracle_pin_{f32,f64}.npz`` hold the inputs (samples) and reference outputs
of the 370 checks of oracle/validate_against_reference.py; ``--oracle-pin``
rewrites only those two files.  The copies in this repository were written
without the reference at hand: each stored output is the output of
oracle/ref_port.py, unchanged since commit 7225f88, where
validate_against_reference.py found it identical to the reference on exactly
these inputs (370 checks, 0 mismatches: 354 bit for bit, the 16 sym_matmul /
sym_det checks to rounding).  Rewrite them with ``--oracle-pin`` where the
reference is installed.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import generators as G          # noqa: E402
from oracle import load_reference           # noqa: E402
from oracle import validate_against_reference  # noqa: E402

BATCH = (3, 8)


def main():
    ref_sym, ref_bat, ref_sugar = load_reference.load()
    sym, dense = {}, {}
    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        for n in range(1, 11):
            k = f"{tag}_n{n}"
            mat = G.spd_packed(BATCH, n, dtype, seed=1000 + n)
            vec = G.vectors(BATCH, n, dtype, seed=2000 + n)
            inp = G.vectors(BATCH, n, dtype, seed=3000 + n)
            reg = G.vectors(BATCH, n, dtype, seed=4000 + n).abs()
            sym[f"{k}_mat"] = mat.numpy()
            sym[f"{k}_vec"] = vec.numpy()
            sym[f"{k}_inp"] = inp.numpy()
            sym[f"{k}_reg"] = reg.numpy()
            sym[f"{k}_matvec"] = ref_sym.sym_matvec(mat, vec).numpy()
            sym[f"{k}_addmatvec"] = (inp + ref_sym.sym_matvec(mat, vec)).numpy()
            sym[f"{k}_submatvec"] = (inp - ref_sym.sym_matvec(mat, vec)).numpy()
            sym[f"{k}_solve"] = ref_sym.sym_solve(mat, vec).contiguous().numpy()
            shifted = mat.clone()
            shifted[..., :n] += reg
            sym[f"{k}_solve_reg"] = ref_sym.sym_solve(shifted, vec).contiguous().numpy()
            sym[f"{k}_invert"] = ref_sym.sym_invert(mat).numpy()
            sym[f"{k}_invert_diag"] = ref_sym.sym_invert(mat, True).numpy()
            sym[f"{k}_full"] = ref_sym.sym_to_full(mat).contiguous().numpy()
            # symmetric indefinite (reference handles these: adjugate / pivoted LU)
            ind = G.sym_indefinite_packed(BATCH, n, dtype, seed=5000 + n)
            sym[f"{k}_ind_mat"] = ind.numpy()
            sym[f"{k}_ind_solve"] = ref_sym.sym_solve(ind, vec).contiguous().numpy()
        # eps exactly as the reference is written (only N == 2 runs)
        mat = G.spd_packed(BATCH, 2, dtype, seed=77)
        vec = G.vectors(BATCH, 2, dtype, seed=78)
        sym[f"{tag}_eps2_mat"] = mat.numpy()
        sym[f"{tag}_eps2_vec"] = vec.numpy()
        sym[f"{tag}_eps2_solve"] = ref_sym.sym_solve(mat, vec, 0.1).contiguous().numpy()

        for n in range(1, 11):
            k = f"{tag}_n{n}"
            a = G.dense_shifted(BATCH, n, dtype, seed=6000 + n)
            b = G.vectors(BATCH, n, dtype, seed=7000 + n)
            s = G.dense_spd(BATCH, n, dtype, seed=8000 + n)
            rhs = G.vectors((*BATCH, n), 3, dtype, seed=9000 + n)
            dense[f"{k}_a"] = a.numpy()
            dense[f"{k}_b"] = b.numpy()
            dense[f"{k}_spd"] = s.numpy()
            dense[f"{k}_rhs"] = rhs.numpy()
            dense[f"{k}_inv"] = ref_bat.batchinv(a).numpy()
            dense[f"{k}_det"] = ref_bat.batchdet(a).numpy()
            dense[f"{k}_matvec"] = ref_bat.batchmatvec(a, b).numpy()
            dense[f"{k}_solve_lu"] = ref_sugar.solvevec(a, b, "lu").numpy()
            dense[f"{k}_solve_chol"] = ref_sugar.solvevec(s, b, "chol").numpy()
            dense[f"{k}_lmdiv_lu"] = ref_sugar.lmdiv(a, rhs, "lu").numpy()
            dense[f"{k}_inv_chol"] = ref_sugar.inv(s, "chol").numpy()
            if n in (2, 3):
                c = a.movedim(-1, 0).movedim(-1, 0)
                fi = ref_bat.inv2 if n == 2 else ref_bat.inv3
                fd = ref_bat.det2 if n == 2 else ref_bat.det3
                dense[f"{k}_closed_inv"] = fi(c).movedim(0, -1).movedim(0, -1).contiguous().numpy()
                dense[f"{k}_closed_det"] = fd(c).contiguous().numpy()
    # "next" rows: sym_outer and sym_matmul straight from the reference
    extra = {}
    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        for n in (1, 2, 3, 5, 10):
            x = G.vectors(BATCH, n, dtype, seed=11000 + n)
            extra[f"{tag}_outer{n}_x"] = x.numpy()
            extra[f"{tag}_outer{n}"] = ref_sym.sym_outer(x).numpy()
        for k, d in ((1, 1), (2, 2), (3, 3), (4, 4), (2, 3), (4, 2), (3, 1), (5, 3), (6, 6)):
            jac = G.vectors((*BATCH, k), d, dtype, seed=12000 + 10 * k + d)
            h = G.spd_packed(BATCH, k, dtype, seed=13000 + k)
            extra[f"{tag}_jhj{k}x{d}_j"] = jac.numpy()
            extra[f"{tag}_jhj{k}x{d}_h"] = h.numpy()
            extra[f"{tag}_jhj{k}x{d}"] = ref_sym.sym_matmul(jac, h).contiguous().numpy()
    np.savez_compressed(os.path.join(HERE, "extra_golden.npz"), **extra)
    np.savez_compressed(os.path.join(HERE, "sym_golden.npz"), **sym)
    np.savez_compressed(os.path.join(HERE, "dense_golden.npz"), **dense)
    write_oracle_pin()
    for f in ("sym_golden.npz", "dense_golden.npz", "extra_golden.npz", "oracle_pin_f32.npz", "oracle_pin_f64.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")


def write_oracle_pin():
    """Inputs and reference outputs of every check of oracle/validate_against_reference.py,
    replayed by tests/test_oracle.py::test_oracle_is_bit_identical_to_reference."""
    rec = {}
    if validate_against_reference.run(record=rec):
        raise SystemExit("the oracle disagrees with the reference: not storing its outputs")
    for tag in ("f32", "f64"):
        part = {k: v for k, v in rec.items() if k.endswith(" " + tag)}
        validate_against_reference.save_pin(os.path.join(HERE, f"oracle_pin_{tag}.npz"), part)


if __name__ == "__main__":
    if sys.argv[1:] == ["--oracle-pin"]:
        write_oracle_pin()
    else:
        main()
