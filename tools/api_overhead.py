#!/usr/bin/env python
"""Host-side cost of one public-API call (tiny batch, so the GPU is idle).

``--root DIR`` times the package of another checkout (e.g. the parent commit's tree, built) with
the same rows, so two versions of the Python layer can be compared in one session.
"""
import argparse, os, sys, time, torch
ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.abspath(ap.parse_args().root))
import nitorch_fastmath_b200 as nfm
dev = "cuda:0"
print(f"# {torch.cuda.get_device_name(dev)}, package {os.path.dirname(nfm.__file__)}")
mat = torch.rand(1024, 6, device=dev) + 3
vec = torch.rand(1024, 3, device=dev)
out = torch.empty_like(vec)
a = torch.rand(1024, 4, 4, device=dev, dtype=torch.float64) + 4 * torch.eye(4, device=dev, dtype=torch.float64)
v4 = torch.rand(1024, 4, device=dev, dtype=torch.float64)
b = torch.rand(1024, 4, 3, device=dev, dtype=torch.float64)
bt = torch.rand(1024, 3, 4, device=dev, dtype=torch.float64)
mat_cf = (torch.rand(6, 1024, device=dev) + 3).t()    # coefficient-first storage viewed coefficient-last
vec_cf = torch.rand(3, 1024, device=dev).t()
j = torch.rand(1024, 3, 3, device=dev) + 2 * torch.eye(3, device=dev)
mat_g = mat.clone().requires_grad_()
gy = torch.rand_like(vec)
def bench(name, f, n=3000):
    for _ in range(100): f()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize()
    print(f"{name:40s} {(time.perf_counter() - t0) / n * 1e6:7.1f} us / call")
bench("sym_solve(mat, vec)", lambda: nfm.sym_solve(mat, vec))
bench("sym_solve(mat, vec, out=out)", lambda: nfm.sym_solve(mat, vec, out=out))
bench("sym_solve(mat, vec, 0.1, out=out)", lambda: nfm.sym_solve(mat, vec, 0.1, out=out))
bench("sym_matvec(mat, vec, out=out)", lambda: nfm.sym_matvec(mat, vec, out=out))
bench("sym_invert(mat)", lambda: nfm.sym_invert(mat))
bench("batchinv(a)", lambda: nfm.batchinv(a))
bench("batchdet(a)", lambda: nfm.batchdet(a))
bench("batchmatvec(a, v)", lambda: nfm.batchmatvec(a, v4))
bench("lmdiv(a, b), k = 3", lambda: nfm.lmdiv(a, b))
bench("rmdiv(b, a), k = 3", lambda: nfm.rmdiv(bt, a))
bench("sym_solve(strided mat, strided vec)", lambda: nfm.sym_solve(mat_cf, vec_cf))
bench("sym_matmul(j, h)", lambda: nfm.sym_matmul(j, mat))
bench("sym_outer(vec)", lambda: nfm.sym_outer(vec))
bench("sym_det(mat)", lambda: nfm.sym_det(mat))
bench("sym_to_full(mat)", lambda: nfm.sym_to_full(mat))
bench("sym_solve_update(x, mat, vec, 0.1)", lambda: nfm.sym_solve_update(vec, mat, vec, 0.1))
bench("sym_matmul_solve(j, h, g)", lambda: nfm.sym_matmul_solve(j, mat, vec))
bench("sym_solve(mat, vec) forward + backward", lambda: nfm.sym_solve(mat_g, vec).backward(gy), n=1000)
bench("torch: mat * 2 (reference point)", lambda: mat * 2)
