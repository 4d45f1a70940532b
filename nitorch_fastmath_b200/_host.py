"""Host-resident operands: chunked H2D -> kernel -> D2H pipeline on the GPU.

When the drop-in functions receive CPU tensors they do NOT compute on the
CPU (there is no CPU path in this package): dense, contiguous operands are
streamed through the GPU with ``nfm_*_host`` (include/nfm.h) and the result
comes back as a CPU tensor, matching the reference's "output lives where the
input lives".  Anything that is not a plain dense batch is uploaded whole,
computed with the device entry point and downloaded.
"""
from __future__ import annotations

import ctypes
import os
import threading
from typing import Optional

import torch

from . import _lib

_DEFAULT_CHUNK_BYTES = int(os.environ.get("NFM_HOST_CHUNK_MB", "16")) << 20   # per pipeline stage, inputs + output
_NBUF = int(os.environ.get("NFM_HOST_NBUF", "3"))


class _DeviceState:
    def __init__(self, device: torch.device):
        self.device = device
        self.streams = [torch.cuda.Stream(device=device) for _ in range(_NBUF)]
        self.stream_array = (ctypes.c_void_p * _NBUF)(*[s.cuda_stream for s in self.streams])
        self.workspace: Optional[torch.Tensor] = None
        self.lock = threading.Lock()   # one pipeline at a time per device: workspace and streams are shared

    def ensure_workspace(self, nbytes: int) -> torch.Tensor:
        if self.workspace is None or self.workspace.numel() < nbytes:
            self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self.workspace


_states = {}
_lock = threading.Lock()


def _state(device: torch.device) -> _DeviceState:
    key = device.index if device.index is not None else torch.cuda.current_device()
    with _lock:
        st = _states.get(key)
        if st is None:
            st = _states[key] = _DeviceState(torch.device("cuda", key))
        return st


def offload_device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError(
            "nitorch_fastmath_b200 has no CPU implementation: CPU tensors are streamed through "
            "a CUDA device, and none is available")
    return torch.device("cuda", torch.cuda.current_device())


def uploaded(call, *tensors: Optional[torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The route for CPU operands that are not streamed: upload ``tensors`` whole to the current
    CUDA device, run ``call`` (the device path) on them and bring its result back, into ``out`` or
    as a new CPU tensor."""
    dev = offload_device()
    r = call(*[None if t is None else t.to(dev, non_blocking=True) for t in tensors])
    if out is not None:
        out.copy_(r)
        return out
    return r.cpu()


def is_plain(t: Optional[torch.Tensor]) -> bool:
    return t is None or (t.device.type == "cpu" and t.is_contiguous())


def chunk_for(dtype: torch.dtype, in_elems: int, out_elems: int, chunk_bytes: int = _DEFAULT_CHUNK_BYTES) -> int:
    es = 8 if dtype == torch.float64 else 4
    chunk = max(1024, chunk_bytes // (es * (in_elems + out_elems)))
    return (chunk // 1024) * 1024


def run_host(fn_name: str, dtype_code: int, dtype: torch.dtype, in_elems: int, out_elems: int, batch: int,
             call, chunk: Optional[int] = None):
    """``call(lib_fn, ws_ptr, ws_bytes, chunk, nbuf, streams)`` -> rc"""
    lib = _lib.load()
    dev = offload_device()
    st = _state(dev)
    if chunk is None:
        chunk = chunk_for(dtype, in_elems, out_elems)
    chunk = max(1, min(chunk, max(batch, 1)))
    nbytes = int(lib.nfm_host_workspace_bytes(dtype_code, chunk, _NBUF, in_elems, out_elems))
    with st.lock, torch.cuda.device(dev):
        ws = st.ensure_workspace(nbytes)
        # the pipeline streams must not start before pending work on the current stream
        cur = torch.cuda.current_stream(dev)
        for s in st.streams:
            s.wait_stream(cur)
        rc = call(getattr(lib, fn_name), ws.data_ptr(), nbytes, chunk, _NBUF, st.stream_array)
    _lib.check(rc, fn_name)
