"""Bandwidth of fp32 7x7 scaled-identity sym_addmatvec (mat (..., 1)) in the large-batch
regime, where the large tile geometry's ring with the addend staged passes the
shared-memory limit: the small tile geometry (TMA path) against the strided kernel,
which took the whole batch before the small geometry was tried.  The strided figure
is forced with an output whose records are padded (not dense), so it is the same
kernel on the same inputs.

    python tools/smem_fallback_timing.py [--batch 8388608] [--reps 50]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, reps):
    for _ in range(3):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8 << 20)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    import nitorch_fastmath_b200 as nfm
    from nitorch_fastmath_b200 import _lib
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"device: {torch.cuda.get_device_name(0)} | {smi}")
    b, n = args.batch, 7
    g = torch.Generator(device="cuda").manual_seed(0)
    mat = torch.rand(b, 1, device="cuda", generator=g) + 0.5
    vec = torch.randn(b, n, device="cuda", generator=g)
    inp = torch.randn(b, n, device="cuda", generator=g)
    out = torch.empty(b, n, device="cuda")
    padded = torch.empty(b, n + 1, device="cuda")[:, :n]
    nbytes = (mat.numel() + vec.numel() + inp.numel() + out.numel()) * 4     # algorithmic traffic

    nfm.sym_addmatvec(inp, mat, vec, out=out)
    shape = _lib.last_launch_shape()
    path = _lib.load().nfm_last_path_was_tma()
    t_tma = timed(lambda: nfm.sym_addmatvec(inp, mat, vec, out=out), args.reps)
    nfm.sym_addmatvec(inp, mat, vec, out=padded)
    assert _lib.load().nfm_last_path_was_tma() == 0
    t_str = timed(lambda: nfm.sym_addmatvec(inp, mat, vec, out=padded), args.reps)
    diff = float(((out - padded).abs() / (inp.abs() + (mat * vec).abs())).max())   # same sums, possibly other roundings
    assert diff < 1e-6, diff
    print(f"batch {b}  ({nbytes / 1e6:.0f} MB algorithmic traffic)")
    print(f"  dispatch: path {path}, launch {shape}")
    print(f"  TMA tile kernel : {t_tma * 1e6:9.1f} us  {nbytes / t_tma / 1e9:7.0f} GB/s")
    print(f"  strided kernel  : {t_str * 1e6:9.1f} us  {nbytes / t_str / 1e9:7.0f} GB/s")


if __name__ == "__main__":
    main()
