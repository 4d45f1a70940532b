"""One process, several GPUs: host-resident batches sharded over the devices.

Every matrix is independent, so the batch axis is cut into contiguous slabs
(``shard.shard_bounds``), one per device; each slab runs its own chunked
H2D -> kernel -> D2H pipeline (``nfm_*_host``) from its own thread (the C
calls release the GIL), and nothing is exchanged between devices.  This is
the single-process counterpart of ``bench.py --gpus N`` (one process per GPU).
"""
from __future__ import annotations

from concurrent.futures import ThreadPoolExecutor
from typing import Callable, Optional, Sequence

import torch
from torch import Tensor

from . import _dispatch as D
from . import sym
from .shard import shard_bounds

__all__ = ["sym_solve_multi", "sym_invert_multi", "sym_matvec_multi"]


def _devices(devices: Optional[Sequence[int]]) -> Sequence[int]:
    if not torch.cuda.is_available():
        raise RuntimeError("nitorch_fastmath_b200 has no CPU implementation and no CUDA device is available")
    if devices is None:
        devices = list(range(torch.cuda.device_count()))
    if len(devices) == 0:
        raise ValueError("no devices given")
    if len(set(devices)) != len(devices):
        raise ValueError(f"duplicate device ids in {list(devices)}: each slab needs its own GPU")
    return devices


def _check_host(*tensors: Optional[Tensor]) -> None:
    for t in tensors:
        if t is not None and (t.device.type != "cpu" or not t.is_contiguous()):
            raise ValueError("the *_multi functions take contiguous CPU tensors (pinned for full speed)")


def _run(devices: Sequence[int], batch: int, work: Callable[[int, int], None]) -> None:
    world = len(devices)

    def job(rank: int) -> None:
        begin, end = shard_bounds(batch, world, rank)
        if end > begin:
            with torch.cuda.device(devices[rank]):   # restored on exit: the caller's current device is untouched
                work(begin, end)

    if world == 1:
        job(0)
        return
    with ThreadPoolExecutor(max_workers=world) as pool:
        for f in [pool.submit(job, r) for r in range(world)]:
            f.result()


def sym_solve_multi(mat: Tensor, vec: Tensor, diag: Optional[Tensor] = None, *, devices: Optional[Sequence[int]] = None,
                    out: Optional[Tensor] = None, method: Optional[str] = None) -> Tensor:
    r"""``mat \ vec`` for CPU tensors ``mat (B, N(N+1)/2)``, ``vec (B, N)`` (and an optional
    per-matrix regulariser ``diag (B, N)``), sharded over ``devices``."""
    _check_host(mat, vec, diag, out)
    D.check_out_shape(out, vec.shape)
    devices = _devices(devices)
    flat_m, flat_v = mat.reshape(-1, mat.shape[-1]), vec.reshape(-1, vec.shape[-1])
    flat_d = diag.reshape(-1, diag.shape[-1]) if diag is not None else None
    if out is None:
        out = torch.empty(vec.shape, dtype=vec.dtype, pin_memory=True)
    flat_o = out.reshape(-1, out.shape[-1])

    def work(b: int, e: int) -> None:
        sym.sym_solve(flat_m[b:e], flat_v[b:e], None if flat_d is None else flat_d[b:e], out=flat_o[b:e], method=method)

    _run(devices, flat_v.shape[0], work)
    return out


def sym_invert_multi(mat: Tensor, diag: bool = False, *, devices: Optional[Sequence[int]] = None,
                     out: Optional[Tensor] = None, method: Optional[str] = None) -> Tensor:
    """Packed inverse (or its diagonal) of CPU ``mat (B, N(N+1)/2)``, sharded over ``devices``."""
    _check_host(mat, out)
    width = D.packed_order(mat.shape[-1]) if diag else mat.shape[-1]
    D.check_out_shape(out, (*mat.shape[:-1], width))
    devices = _devices(devices)
    flat_m = mat.reshape(-1, mat.shape[-1])
    if out is None:
        out = torch.empty((*mat.shape[:-1], width), dtype=mat.dtype, pin_memory=True)
    flat_o = out.reshape(-1, out.shape[-1])

    def work(b: int, e: int) -> None:
        sym.sym_invert(flat_m[b:e], diag, out=flat_o[b:e], method=method)

    _run(devices, flat_m.shape[0], work)
    return out


def sym_matvec_multi(mat: Tensor, vec: Tensor, *, devices: Optional[Sequence[int]] = None,
                     out: Optional[Tensor] = None) -> Tensor:
    """``mat @ vec`` for CPU tensors, sharded over ``devices``."""
    _check_host(mat, vec, out)
    D.check_out_shape(out, vec.shape)
    devices = _devices(devices)
    flat_m, flat_v = mat.reshape(-1, mat.shape[-1]), vec.reshape(-1, vec.shape[-1])
    if out is None:
        out = torch.empty(vec.shape, dtype=torch.promote_types(mat.dtype, vec.dtype), pin_memory=True)
    flat_o = out.reshape(-1, out.shape[-1])

    def work(b: int, e: int) -> None:
        sym.sym_matvec(flat_m[b:e], flat_v[b:e], out=flat_o[b:e])

    _run(devices, flat_v.shape[0], work)
    return out
