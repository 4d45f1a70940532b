#!/usr/bin/env python
"""Forward / backward time of the differentiable packed-symmetric routines, and the
bandwidth of the backward kernels (nfm_sym_outer2, nfm_sym_invert_backward,
nfm_sym_det_backward) against the measured copy peak.  ``--dense`` measures the dense
routines instead (batchdet, batchinv, solvevec, lmdiv, rmdiv; nfm_batch_inv_backward,
nfm_batch_det_backward, nfm_batch_outer, nfm_batch_tsolve) and autograd through torch's
own linalg functions on the same GPU.  ``--gn`` measures the Gauss-Newton builders
(sym_matmul, sym_matmul_solve, sym_solve_update, sym_outer, sym_to_full;
nfm_sym_matmul_backward, nfm_sym_outer_backward, nfm_sym_to_full_backward) and autograd
through the oracle on the same GPU.

CUDA events around many calls after a warm-up; every field is larger than the
126 MB L2 of a B200 (except the tiny-batch gate-cost rows, which time host work).
Prints a report; ``--out FILE`` also writes it there."""
import argparse
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nitorch_fastmath_b200 as nfm  # noqa: E402
from nitorch_fastmath_b200 import _autograd as A  # noqa: E402
from nitorch_fastmath_b200 import _lib, sym  # noqa: E402
from oracle import generators as G  # noqa: E402
from oracle import ref_port as P  # noqa: E402

DEV = "cuda:0"
LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def ev_time(fn, reps=20, warm=3):
    """Mean milliseconds per call of fn() (CUDA events, after warm-up)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_peak():
    x = torch.empty(1 << 29, dtype=torch.float32, device=DEV)   # 2 GiB
    y = torch.empty_like(x)
    ms = ev_time(lambda: y.copy_(x), reps=20)
    return 2 * x.numel() * 4 / ms / 1e6   # GB/s


def field(shape, n, dtype, seed):
    """SPD packed field built on the GPU: (G G^T + n I) from a seeded normal field."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    a = torch.randn(*shape, n, n, device=DEV, dtype=dtype, generator=g) * 0.3
    full = a @ a.mT
    full.diagonal(0, -1, -2).add_(n)
    iu = torch.triu_indices(n, n, 1, device=DEV)
    m = torch.cat([full.diagonal(0, -1, -2), full[..., iu[0], iu[1]]], -1).contiguous()
    del a, full
    return m


def vecs(shape, n, dtype, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.randn(*shape, n, device=DEV, dtype=dtype, generator=g)


def fwd_bwd(name, fwd, leaves, gout):
    """Forward with grad-requiring inputs, and the backward alone (graph rebuilt per call, untimed)."""
    t_plain = ev_time(lambda: fwd(*[t.detach() for t in leaves]))
    t_fwd = ev_time(lambda: fwd(*leaves))
    out = [None]

    def bwd():
        torch.autograd.grad(out[0], leaves, gout)

    for _ in range(3):
        out[0] = fwd(*leaves)
        bwd()
    torch.cuda.synchronize()
    total = 0.0
    reps = 10
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        out[0] = fwd(*leaves)
        torch.cuda.synchronize()
        a.record()
        bwd()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    say(f"{name:44s} forward no-grad {t_plain:8.3f} ms   forward with grad {t_fwd:8.3f} ms   backward {total / reps:8.3f} ms")


def dense_field(batch, n, dtype, seed, spd=False):
    """randn + n I (or G G^T + n I with ``spd``), built on the GPU."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    a = torch.randn(*batch, n, n, device=DEV, dtype=dtype, generator=g)
    if spd:
        a = a @ a.mT * 0.1
    a.diagonal(0, -1, -2).add_(n)
    return a


def dense(peak):
    lib = _lib.load()
    f32, f64 = torch.float32, torch.float64
    say("== dense routines: forward / backward, fields larger than L2 ==")
    cube = (256, 256, 256)
    a = dense_field(cube, 3, f32, 1)
    fwd_bwd("batchdet 256^3 3x3 fp32", nfm.batchdet, [a.requires_grad_()], vecs(cube[:-1], cube[-1], f32, 2))
    fwd_bwd("torch.linalg.det 256^3 3x3 fp32", torch.linalg.det, [a], vecs(cube[:-1], cube[-1], f32, 2))
    gi = dense_field(cube, 3, f32, 3)
    fwd_bwd("batchinv 256^3 3x3 fp32", nfm.batchinv, [a], gi)
    fwd_bwd("torch.linalg.inv 256^3 3x3 fp32", torch.linalg.inv, [a], gi)
    del a, gi
    torch.cuda.empty_cache()
    b16 = (16 << 20,)
    a = dense_field(b16, 4, f64, 1).requires_grad_()
    gi = dense_field(b16, 4, f64, 2)
    fwd_bwd("batchinv 16M 4x4 fp64", nfm.batchinv, [a], gi)
    fwd_bwd("torch.linalg.inv 16M 4x4 fp64", torch.linalg.inv, [a], gi)
    del gi
    v, g = vecs(b16, 4, f64, 3).requires_grad_(), vecs(b16, 4, f64, 4)
    fwd_bwd("solvevec 16M 4x4 fp64 (d mat, d vec)", nfm.solvevec, [a, v], g)
    fwd_bwd("torch.linalg.solve 16M 4x4 fp64 (d mat, d vec)", lambda a, v: torch.linalg.solve(a, v), [a, v], g)
    del a, v, g
    torch.cuda.empty_cache()
    b4 = (4 << 20,)
    a = dense_field(b4, 4, f32, 1).requires_grad_()
    for k in (3, 8):
        b, g = vecs(b4 + (4,), k, f32, 2).requires_grad_(), vecs(b4 + (4,), k, f32, 3)
        fwd_bwd(f"lmdiv 4M 4x4 k={k} fp32", nfm.lmdiv, [a, b], g)
        fwd_bwd(f"torch.linalg.solve 4M 4x4 k={k} fp32", torch.linalg.solve, [a, b], g)
    x, g = vecs(b4 + (3,), 4, f32, 4).requires_grad_(), vecs(b4 + (3,), 4, f32, 5)
    fwd_bwd("rmdiv 4M 3 rows x 4x4 fp32", nfm.rmdiv, [x, a], g)
    fwd_bwd("torch.linalg.solve(left=False) 4M 3 rows fp32", lambda x, a: torch.linalg.solve(a, x, left=False), [x, a], g)
    del a, b, g, x
    torch.cuda.empty_cache()

    say()
    say("== dense backward kernels: algorithmic bytes / time, against the copy peak ==")
    say("   inverse backward 3n^2 s, det backward (2n^2+1) s, outer (2nk+n^2) s, transposed solve (n^2+2nk) s")
    say(f"{'kernel':44s} {'dtype':8s} {'batch':>10s} {'us':>10s} {'GB/s':>8s} {'of peak':>8s} path")
    for dtype in (f32, f64):
        s = torch.tensor([], dtype=dtype).element_size()
        for n in (3, 4, 6, 8, 10):
            batch = int(2e9 // (3 * n * n * s))        # ~2 GB of traffic per call
            y, gm = dense_field((batch,), n, dtype, 1), vecs((batch, n), n, dtype, 2)
            rows = [("inverse backward n=%d" % n, lambda: A.dense_inv_backward(y, gm, False), 3 * n * n),
                    ("inverse backward chol n=%d" % n, lambda: A.dense_inv_backward(y, gm, True), 3 * n * n)]
            gd = gm[:, 0, 0].contiguous()
            rows.append(("det backward n=%d" % n, lambda: A.dense_det_backward(y, gd), 2 * n * n + 1))
            for label, fn, nb in rows:
                ms = ev_time(fn)
                path = lib.nfm_last_path_was_tma()
                gbs = nb * s * batch / ms / 1e6
                say(f"{label:44s} {str(dtype)[6:]:8s} {batch:10d} {ms * 1e3:10.1f} {gbs:8.0f} {gbs / peak:8.2f} {path}")
            del gm, gd
            for k in (1, 3):
                u, w = vecs((batch, n), k, dtype, 3), vecs((batch, n), k, dtype, 4)
                for label, fn, nb in (("outer n=%d k=%d" % (n, k), lambda: A.dense_outer(u, w, False, False, -1), 2 * n * k + n * n),
                                      ("transposed solve lu n=%d k=%d" % (n, k), lambda: A.dense_tsolve(y, u, False, _lib.ALGO_LU),
                                       n * n + 2 * n * k)):
                    ms = ev_time(fn)
                    path = lib.nfm_last_path_was_tma()
                    gbs = nb * s * batch / ms / 1e6
                    say(f"{label:44s} {str(dtype)[6:]:8s} {batch:10d} {ms * 1e3:10.1f} {gbs:8.0f} {gbs / peak:8.2f} {path}")
                del u, w
            del y
            torch.cuda.empty_cache()


def jacobian(shape, k, d, dtype, seed):
    """0.1 randn plus ones on the leading diagonal, built on the GPU."""
    j = vecs(shape + (k,), d, dtype, seed) * 0.1
    j[..., range(min(k, d)), range(min(k, d))] += 1.0
    return j


def gn(peak):
    lib = _lib.load()
    f32 = torch.float32
    say("== Gauss-Newton builders: forward / backward (all inputs), fp32, fields larger than L2 ==")
    for side, k, d in ((160, 10, 3), (192, 6, 6), (256, 3, 3)):
        shape = (side, side, side)
        mode1 = k == d and k <= 3
        kh, ko = (d, k) if mode1 else (k, d)
        j, h = jacobian(shape, k, d, f32, 1).requires_grad_(), field(shape, kh, f32, 2).requires_grad_()
        tag = f"{side}^3 k={k} d={d}" + (" (mode 1)" if mode1 else "")
        fwd_bwd(f"sym_matmul {tag}", nfm.sym_matmul, [j, h], vecs(shape, ko * (ko + 1) // 2, f32, 3))
        g0 = vecs(shape, ko, f32, 4).requires_grad_()
        fwd_bwd(f"sym_matmul_solve {tag}", lambda j, h, g0: nfm.sym_matmul_solve(j, h, g0, 1.0), [j, h, g0], vecs(shape, ko, f32, 5))
        del j, h, g0
        torch.cuda.empty_cache()
    shape = (256, 256, 256)
    x, m, v = vecs(shape, 3, f32, 1).requires_grad_(), field(shape, 3, f32, 2).requires_grad_(), vecs(shape, 3, f32, 3).requires_grad_()
    gs = vecs(shape, 3, f32, 4)
    fwd_bwd("sym_solve_update 256^3 N=3", lambda x, m, v: nfm.sym_solve_update(x, m, v, 0.1, 0.5), [x, m, v], gs)
    fwd_bwd("sym_outer 256^3 N=3", nfm.sym_outer, [x], vecs(shape, 6, f32, 5))
    del x, m, v, gs
    torch.cuda.empty_cache()
    shape = (192, 192, 192)
    m = field(shape, 6, f32, 1).requires_grad_()
    fwd_bwd("sym_to_full 192^3 N=6", nfm.sym_to_full, [m], vecs(shape + (6,), 6, f32, 2))
    del m
    torch.cuda.empty_cache()

    say()
    say("== autograd through the oracle (eager torch, what the reference does), same GPU, fp32 ==")
    shape = (192, 192, 192)
    j, h = jacobian(shape, 6, 6, f32, 1).requires_grad_(), field(shape, 6, f32, 2).requires_grad_()
    fwd_bwd("oracle sym_matmul 192^3 k=6 d=6", P.sym_matmul, [j, h], vecs(shape, 21, f32, 3))
    del j, h
    torch.cuda.empty_cache()
    shape = (256, 256, 256)
    j, h, g0 = jacobian(shape, 3, 3, f32, 1).requires_grad_(), field(shape, 3, f32, 2).requires_grad_(), vecs(shape, 3, f32, 4).requires_grad_()
    one = torch.ones(3, device=DEV, dtype=f32)     # the oracle takes a float regulariser on the CPU only
    fwd_bwd("oracle sym_matmul_solve 256^3 k=d=3 (mode 1)", lambda j, h, g0: P.sym_solve(P.sym_matmul(j, h), g0, one),
            [j, h, g0], vecs(shape, 3, f32, 5))
    del j, h
    m, x = field(shape, 3, f32, 2).requires_grad_(), vecs(shape, 3, f32, 1).requires_grad_()
    fwd_bwd("oracle sym_solve_update 256^3 N=3", lambda x, m, v: x - 0.5 * P.sym_solve(m, v, 0.1 * one), [x, m, g0], vecs(shape, 3, f32, 6))
    fwd_bwd("oracle sym_outer 256^3 N=3", P.sym_outer, [x], vecs(shape, 6, f32, 5))
    del m, x, g0
    torch.cuda.empty_cache()
    shape = (192, 192, 192)
    m = field(shape, 6, f32, 1).requires_grad_()
    fwd_bwd("oracle sym_to_full 192^3 N=6", P.sym_to_full, [m], vecs(shape + (6,), 6, f32, 2))
    del m
    torch.cuda.empty_cache()

    say()
    say("== Gauss-Newton backward kernels: algorithmic bytes / time, against the copy peak ==")
    say("   matmul backward (J, H, g in; dJ and / or dH out), outer backward (2N + NN) s, to_full backward (N^2 + NN) s")
    say(f"{'kernel':44s} {'dtype':8s} {'batch':>10s} {'us':>10s} {'GB/s':>8s} {'of peak':>8s} path")

    def row(label, dtype, batch, fn, nelem):
        ms = ev_time(fn)
        path = lib.nfm_last_path_was_tma()
        gbs = nelem * torch.tensor([], dtype=dtype).element_size() * batch / ms / 1e6
        say(f"{label:44s} {str(dtype)[6:]:8s} {batch:10d} {ms * 1e3:10.1f} {gbs:8.0f} {gbs / peak:8.2f} {path}")

    for dtype in (torch.float32, torch.float64):
        s = torch.tensor([], dtype=dtype).element_size()
        for k, d in ((3, 3), (6, 6), (10, 3), (10, 10)):
            mode1 = k == d and k <= 3
            kh, ko = (d, k) if mode1 else (k, d)
            hh, oo = kh * (kh + 1) // 2, ko * (ko + 1) // 2
            batch = int(2e9 // ((2 * k * d + 2 * hh + oo) * s))
            j, h, g = jacobian((batch,), k, d, dtype, 1), field((batch,), kh, dtype, 2), vecs((batch,), oo, dtype, 3)
            for which, name, nout in ((1, "dJ", k * d), (2, "dH", hh), (3, "dJ+dH", k * d + hh)):
                row(f"matmul backward k={k} d={d} {name}", dtype, batch, lambda: A.matmul_backward(j, h, g, which),
                    k * d + hh + oo + nout)
            del j, h, g
            torch.cuda.empty_cache()
        for n in (3, 6, 10):
            nn = n * (n + 1) // 2
            batch = int(2e9 // ((2 * n + nn) * s))
            x, g = vecs((batch,), n, dtype, 1), vecs((batch,), nn, dtype, 2)
            row(f"outer backward N={n}", dtype, batch, lambda: A.outer_backward(x, g), 2 * n + nn)
            del x, g
            batch = int(2e9 // ((n * n + nn) * s))
            g = vecs((batch, n), n, dtype, 3)
            row(f"to_full backward N={n}", dtype, batch, lambda: A.to_full_backward(g), n * n + nn)
            del g
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--out", default=None)
    ap.add_argument("--dense", action="store_true", help="measure the dense routines instead of the packed ones")
    ap.add_argument("--gn", action="store_true", help="measure the Gauss-Newton builders instead of the packed solves")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grad_timing needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    say(f"GPU 0: {q}   ({torch.cuda.get_device_name(0)}; torch {torch.__version__})")
    peak = copy_peak()
    say(f"measured copy peak (2 GiB device-to-device copy, read + write bytes): {peak:.0f} GB/s")
    say()
    if args.dense or args.gn:
        (dense if args.dense else gn)(peak)
        if args.out:
            with open(args.out, "w") as fh:
                fh.write("\n".join(LINES) + "\n")
        return
    say("== forward / backward, fp32, fields larger than L2 ==")
    f32 = torch.float32
    for side, n in ((256, 3), (192, 6), (160, 10)):
        shape = (side, side, side)
        m, v, g = field(shape, n, f32, 1), vecs(shape, n, f32, 2), vecs(shape, n, f32, 3)
        fwd_bwd(f"sym_solve {side}^3 N={n} (d mat, d vec)", lambda m, v: nfm.sym_solve(m, v),
                [m.requires_grad_(), v.requires_grad_()], g)
        del m, v, g
        torch.cuda.empty_cache()
    shape, n = (192, 192, 192), 6
    nn = n * (n + 1) // 2
    m = field(shape, n, f32, 1)
    fwd_bwd(f"sym_invert 192^3 N={n}", lambda m: nfm.sym_invert(m), [m.requires_grad_()], vecs(shape, nn, f32, 4))
    fwd_bwd(f"sym_invert(diag=True) 192^3 N={n}", lambda m: nfm.sym_invert(m, True), [m], vecs(shape, n, f32, 4))
    fwd_bwd(f"sym_det 192^3 N={n}", lambda m: nfm.sym_det(m), [m], vecs(shape, 1, f32, 5)[..., 0])
    del m
    torch.cuda.empty_cache()

    say()
    say("== N=3 reference: autograd through the oracle (eager torch) on the same GPU, 256^3 fp32 ==")
    shape, n = (256, 256, 256), 3
    m, v, g = field(shape, n, f32, 1), vecs(shape, n, f32, 2), vecs(shape, n, f32, 3)
    fwd_bwd("oracle sym_solve 256^3 N=3", lambda m, v: P.sym_solve(m, v), [m.requires_grad_(), v.requires_grad_()], g)
    fwd_bwd("nfm    sym_solve 256^3 N=3", lambda m, v: nfm.sym_solve(m, v), [m, v], g)
    del m, v, g
    torch.cuda.empty_cache()

    say()
    say("== backward kernels: algorithmic bytes / time, against the copy peak ==")
    say(f"{'kernel':44s} {'dtype':8s} {'batch':>10s} {'us':>10s} {'GB/s':>8s} {'of peak':>8s} path")
    lib = _lib.load()
    for dtype in (torch.float32, torch.float64):
        s = torch.tensor([], dtype=dtype).element_size()
        for n in (3, 6, 10):
            nn = n * (n + 1) // 2
            batch = int(2e9 // ((2 * nn + n) * s))        # ~2 GB of traffic per call
            u, w = vecs((batch,), n, dtype, 1), vecs((batch,), n, dtype, 2)
            for lname, layout, ln in (("S", _lib.LAYOUT_SYM, nn), ("D", _lib.LAYOUT_DIAG, n), ("E", _lib.LAYOUT_SCALED_IDENTITY, 1)):
                if lname != "S" and n != 6:
                    continue
                ms = ev_time(lambda: A.outer2(u, w, layout, -1))
                path = lib.nfm_last_path_was_tma()
                gbs = (2 * n + ln) * s * batch / ms / 1e6
                say(f"{'outer2 N=%d layout %s' % (n, lname):44s} {str(dtype)[6:]:8s} {batch:10d} {ms * 1e3:10.1f} {gbs:8.0f} {gbs / peak:8.2f} {path}")
            del u, w
            b = field((batch // 2,), n, dtype, 3)
            gp, gd, gs = vecs((batch // 2,), nn, dtype, 4), vecs((batch // 2,), n, dtype, 5), vecs((batch // 2,), 1, dtype, 6)[:, 0]
            for label, fn, nbytes in (("invert backward N=%d" % n, lambda: A.invert_backward(b, gp, False), 3 * nn),
                                      ("invert backward diag_only N=%d" % n, lambda: A.invert_backward(b, gd, True), 2 * nn + n),
                                      ("det backward N=%d" % n, lambda: A.det_backward(b, gs), 2 * nn + 1)):
                ms = ev_time(fn)
                path = lib.nfm_last_path_was_tma()
                gbs = nbytes * s * (batch // 2) / ms / 1e6
                say(f"{label:44s} {str(dtype)[6:]:8s} {batch // 2:10d} {ms * 1e3:10.1f} {gbs:8.0f} {gbs / peak:8.2f} {path}")
            del b, gp, gd, gs
            torch.cuda.empty_cache()

    say()
    say("== cost of the no-grad gate: public call vs the implementation behind it (1024 x N=3 fp32, host-bound) ==")
    m, v = field((1024,), 3, f32, 1), vecs((1024,), 3, f32, 2)
    pairs = [("sym_solve", lambda: nfm.sym_solve(m, v), lambda: sym._solve(m, v)),
             ("sym_matvec", lambda: nfm.sym_matvec(m, v), lambda: sym._matvec(None, m, v, 0, None, None)),
             ("sym_invert", lambda: nfm.sym_invert(m), lambda: sym._invert(m)),
             ("sym_det", lambda: nfm.sym_det(m), lambda: sym._det(m))]
    for name, pub, impl in pairs:
        res = []
        for f in (pub, impl, pub, impl):       # alternate, keep the better of two rounds
            for _ in range(200):
                f()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5000):
                f()
            torch.cuda.synchronize()
            res.append((time.perf_counter() - t0) / 5000 * 1e6)
        say(f"{name:12s} public {min(res[0], res[2]):6.2f} us/call   implementation {min(res[1], res[3]):6.2f} us/call   "
            f"gate {min(res[0], res[2]) - min(res[1], res[3]):+5.2f} us")
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
