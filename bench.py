#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched small-matrix hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload sym_solve3|sym_solve6|sym_invert6|sym_solve10|dense_inv4_f64|...]
                    [--dump-outputs DIR]

Metric (BASELINE.json): batched sym-solve matrices/s and achieved HBM GB/s
vs peak.  A "step" is one pass of the hot path over the whole workload:
the default workload is BASELINE.json configs[1], the 256^3-voxel 3x3
compact-symmetric solve in fp32 (16 777 216 matrices, 48 B each).

  value   whole-job matrices/s with operands resident in HBM, CUDA events on
          the launch stream, K back-to-back launches through the C ABI.  The K
          calls are captured once in a CUDA graph and ONE replay is timed
          (--launch graph, the default: with 16 us launches at 8 GPUs the Python
          loop itself was 8 % of the region); --launch eager times K ctypes calls.
  e2e     the same metric through the public API with HOST (pinned) operands:
          chunked H2D -> kernel -> D2H inside the timed region.
  N > 1   strong scaling (north star): the batch is split into N contiguous
          slabs, one process per GPU, no data-path collective; torch.distributed
          is used only for the barrier and the max-over-ranks of the time.

One JSON line on stdout (rank 0).  With --impl reference the reference's own CPU
implementation (unmodified, from baseline/_ref -- kind "reference"; the pinned
oracle port only if it cannot be imported) is timed on the host cores.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

L2_BYTES = 126 << 20
DUMP_BUDGET = 60 << 20      # --dump-outputs: bytes written per invocation, all workloads and ranks together
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback

# name -> (kind, n, dtype, voxels-per-side or batch, description)
WORKLOADS = {
    "sym_solve3": dict(kind="sym_solve", n=3, dtype="f32", batch=256 ** 3,
                       desc="256^3-voxel 3x3 compact-sym solve fp32 (BASELINE.json configs[1])"),
    "sym_solve6": dict(kind="sym_solve", n=6, dtype="f32", batch=192 ** 3,
                       desc="192^3-voxel 6x6 compact-sym solve fp32 (configs[2])"),
    "sym_invert6": dict(kind="sym_invert", n=6, dtype="f32", batch=192 ** 3,
                        desc="192^3-voxel 6x6 compact-sym invert fp32 (configs[2])"),
    "sym_solve10": dict(kind="sym_solve", n=10, dtype="f32", batch=160 ** 3,
                        desc="160^3-voxel 10x10 compact-sym solve fp32 (configs[4])"),
    "sym_matvec3": dict(kind="sym_matvec", n=3, dtype="f32", batch=256 ** 3,
                        desc="256^3-voxel 3x3 compact-sym matvec fp32"),
    "sym_solve3_1m": dict(kind="sym_solve", n=3, dtype="f32", batch=1_000_000,
                          desc="1M 3x3 compact-sym solve fp32 (configs[0])"),
    "dense_inv4_f64": dict(kind="batch_inv", n=4, dtype="f64", batch=64 << 20,
                           desc="64M general 4x4 inverse fp64 (configs[3])"),
    "dense_det4_f64": dict(kind="batch_det", n=4, dtype="f64", batch=64 << 20,
                           desc="64M general 4x4 det fp64 (configs[3])"),
    "dense_solve4_f64": dict(kind="batch_solve", n=4, dtype="f64", batch=64 << 20,
                             desc="64M general 4x4 LU solve fp64 (configs[3])"),
}


def record_lengths(kind: str, n: int):
    """(input record lengths, output record length) in elements."""
    nn = n * (n + 1) // 2
    return {
        "sym_solve": ([nn, n], n),
        "sym_matvec": ([nn, n], n),
        "sym_invert": ([nn], nn),
        "batch_inv": ([n * n], n * n),
        "batch_det": ([n * n], 1),
        "batch_solve": ([n * n, n], n),
    }[kind]


def algorithmic_bytes(kind: str, n: int, esize: int) -> int:
    """Minimum HBM traffic per matrix (SURVEY.md section 8d)."""
    ins, out = record_lengths(kind, n)
    return (sum(ins) + out) * esize


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload: str):
    """dram__bytes_read+write per launch from the committed ncu capture, if any."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


# --------------------------------------------------------------------------
# synthetic data, generated on the device (seeded), shaped like the workload
# --------------------------------------------------------------------------

def make_inputs(kind: str, n: int, dtype: torch.dtype, batch: int, device, seed: int):
    g = torch.Generator(device=device).manual_seed(seed)
    if kind.startswith("sym"):
        out = []
        chunk = 1 << 21
        for b0 in range(0, batch, chunk):
            b = min(chunk, batch - b0)
            a = torch.randn(b, n, n, device=device, dtype=dtype, generator=g)
            full = a @ a.transpose(-1, -2)
            full.diagonal(0, -1, -2).add_(n)
            iu = torch.triu_indices(n, n, 1, device=device)
            out.append(torch.cat([full.diagonal(0, -1, -2), full[..., iu[0], iu[1]]], -1))
        mat = torch.cat(out).contiguous()
        if kind == "sym_invert":
            return [mat]
        return [mat, torch.randn(batch, n, device=device, dtype=dtype, generator=g)]
    a = torch.randn(batch, n, n, device=device, dtype=dtype, generator=g)
    a.diagonal(0, -1, -2).add_(10)
    if kind == "batch_solve":
        return [a, torch.randn(batch, n, device=device, dtype=dtype, generator=g)]
    return [a]


def operand_set_count(set_bytes: int) -> int:
    """Distinct operand sets the steps rotate through: enough that consecutive steps never
    find their data in L2 (one if a set is already several times L2)."""
    return 1 if set_bytes >= 3 * L2_BYTES else min(8, math.ceil(3 * L2_BYTES / max(set_bytes, 1)))


def operand_seed(rank: int, s: int) -> int:
    """``make_inputs`` seed of operand set ``s`` of ``rank``."""
    return 1000 * rank + s


def timed_set(warmup: int, step: int, nsets: int) -> int:
    """Operand set of timed step ``step`` (0-based): the rotation continues from the warm-up."""
    return (warmup + step) % nsets


ALGOS = {"auto": 0, "ldl": 1, "lu": 2, "warp": 3}


def abi_launcher(lib, kind: str, n: int, code: int, batch: int, ins, out, stream: int, algo: int = 0):
    """Zero-argument callable = one pass of the hot path through the C ABI
    (include/nfm.h), with every argument evaluated once up front."""
    import functools
    lens, olen = record_lengths(kind, n)
    p = [t.data_ptr() for t in ins]
    o = out.data_ptr()
    if kind == "sym_solve":
        return functools.partial(lib.nfm_sym_solve, code, n, 2, algo, batch, p[0], lens[0], p[1], lens[1], None, 0, o, olen, stream)
    if kind == "sym_matvec":
        return functools.partial(lib.nfm_sym_matvec, code, n, 2, batch, p[0], lens[0], p[1], lens[1], None, 0, 0, o, olen, stream)
    if kind == "sym_invert":
        return functools.partial(lib.nfm_sym_invert, code, n, algo, 0, batch, p[0], lens[0], o, olen, stream)
    if kind == "batch_inv":
        return functools.partial(lib.nfm_batch_inv, code, n, 0, 1, batch, p[0], lens[0], o, olen, stream)
    if kind == "batch_det":
        return functools.partial(lib.nfm_batch_det, code, n, batch, p[0], lens[0], o, olen, stream)
    if kind == "batch_solve":
        return functools.partial(lib.nfm_batch_solve, code, n, 1, 2, batch, p[0], lens[0], p[1], lens[1], o, olen, stream)
    raise ValueError(kind)


def api_call(kind: str, ins, out):
    """The call a user makes (public drop-in API)."""
    from nitorch_fastmath_b200 import batched, sugar, sym
    if kind == "sym_solve":
        return sym.sym_solve(ins[0], ins[1], out=out)
    if kind == "sym_matvec":
        return sym.sym_matvec(ins[0], ins[1], out=out)
    if kind == "sym_invert":
        return sym.sym_invert(ins[0], out=out)
    if kind == "batch_inv":
        return batched.batchinv(ins[0], out=out)
    if kind == "batch_det":
        return batched.batchdet(ins[0], out=out)
    if kind == "batch_solve":
        return sugar.solvevec(ins[0], ins[1], out=out)
    raise ValueError(kind)


_REFERENCE = None


def reference_impl():
    """(kind label, module-like namespace of callables): the reference's OWN code when it
    can be imported (baseline/_ref, installed by oracle/install_reference.py, or the
    directory NFM_REFERENCE_ROOT names), else the oracle port."""
    global _REFERENCE
    if _REFERENCE is None:
        try:
            from oracle import load_reference as L
            if not L.available():
                raise RuntimeError("no reference install")
            ref_sym, ref_batched, ref_sugar = L.load()
            _REFERENCE = ("reference", {
                "sym_solve": ref_sym.sym_solve, "sym_matvec": ref_sym.sym_matvec, "sym_invert": ref_sym.sym_invert,
                "batch_inv": ref_batched.batchinv, "batch_det": ref_batched.batchdet, "batch_solve": ref_sugar.solvevec,
            }, "nitorch_fastmath (unmodified, %s): _impl/sym.py, _impl/batched.py, sugar.py" % L.REFERENCE_ROOT)
        except Exception as exc:  # noqa: BLE001 -- any import problem -> the pinned port
            from oracle import ref_port as P
            _REFERENCE = ("port", {
                "sym_solve": P.sym_solve, "sym_matvec": P.sym_matvec, "sym_invert": P.sym_invert,
                "batch_inv": P.batchinv, "batch_det": P.batchdet, "batch_solve": P.solvevec,
            }, "oracle/ref_port.py = the reference's torch-CPU algorithm (reference not importable: %s)" % exc)
    return _REFERENCE


def oracle_call(kind: str, ins):
    return reference_impl()[1][kind](*ins)


def bind_to_gpu_cpus(index: int):
    """Pin this rank to the CPUs NVML reports as local to its GPU, so that the
    pinned host buffers of the e2e path are first-touched on the GPU's NUMA node
    (matters when several ranks stream over PCIe at once)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# --------------------------------------------------------------------------
# clocks during the timed region (NVML)
# --------------------------------------------------------------------------

_SAMPLER_SRC = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
period = float(sys.argv[2])
print("max", nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM), flush=True)
while True:
    t = time.time()
    try:
        print(t, nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksThrottleReasons(h), flush=True)
    except Exception:
        pass
    time.sleep(period)
"""


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, polled from NVML by a separate
    PROCESS (a sampling thread in this process would fight the launch loop for the GIL: with
    20 steps of 16 us the timed region is 0.3 ms long).  Start it well before the region
    (``start()``), bracket the region with ``with sampler:``; samples are matched by wall clock.
    Regions shorter than the NVML polling period also take the samples just before / after."""
    REASONS = {
        0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
        0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
        0x100: "display_clock_setting",
    }

    def __init__(self, index: int, period: float = 0.002):
        import subprocess
        import tempfile
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._t0 = self._t1 = None
        self._out = tempfile.NamedTemporaryFile("w+", suffix=".clocks", delete=False)
        try:
            self._proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(index), str(period)],
                                          stdout=self._out, stderr=subprocess.DEVNULL)
        except Exception:
            self._proc = None

    def wait_ready(self, timeout: float = 10.0):
        """Block until the sampler process has produced its first sample (it imports pynvml first)."""
        t_end = time.time() + timeout
        while self._proc is not None and time.time() < t_end:
            if os.path.getsize(self._out.name) > 40:
                return
            time.sleep(0.01)

    def __enter__(self):
        self._t0 = time.time()
        return self

    def __exit__(self, *exc):
        self._t1 = time.time()
        time.sleep(0.003)          # let the sampler take one more sample after the region
        if self._proc is not None:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=5)
            except Exception:
                self._proc.kill()
        rows = []
        try:
            with open(self._out.name) as f:
                for line in f:
                    p = line.split()
                    if len(p) == 2 and p[0] == "max":
                        self.max_mhz = int(p[1])
                    elif len(p) == 3:
                        rows.append((float(p[0]), int(p[1]), int(p[2])))
            os.unlink(self._out.name)
        except Exception:
            pass
        inside = [r for r in rows if self._t0 <= r[0] <= self._t1]
        if len(inside) < 3:        # very short region: the samples that bracket it
            before = [r for r in rows if r[0] < self._t0][-2:]
            after = [r for r in rows if r[0] > self._t1][:2]
            inside = before + inside + after
        for _, mhz, mask in inside:
            self.samples.append(mhz)
            for bit, name in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------

def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline(kind, n, dtype, batch, steps=3, warmup=1, budget_s=20.0):
    """The reference's CPU implementation (its own code from baseline/_ref when
    importable, else the pinned oracle port) on all host cores, on a bounded sample of the
    workload: the sample is sized from a calibration run so that
    (warmup + steps) passes take about ``budget_s`` seconds."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen_dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    cal = min(batch, 1 << 20)
    ins = [t.cpu() for t in make_inputs(kind, n, dtype, cal, gen_dev, seed=0)]
    oracle_call(kind, [t[:4096] for t in ins])            # TorchScript-free, but warms the allocator
    t0 = time.perf_counter()
    oracle_call(kind, ins)
    per_matrix = (time.perf_counter() - t0) / cal
    sample = int(budget_s / (steps + warmup) / per_matrix)
    sample = max(min(sample, batch), min(batch, 1 << 16))
    if sample != cal:
        ins = [t.cpu() for t in make_inputs(kind, n, dtype, sample, gen_dev, seed=0)]
    for _ in range(warmup):
        oracle_call(kind, ins)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        oracle_call(kind, ins)
        times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    # one single-thread figure for context (SURVEY.md section 8d), on a slice of the sample
    single = None
    try:
        small = [t[: min(sample, 1 << 21)] for t in ins]
        torch.set_num_threads(1)
        oracle_call(kind, small)
        t0 = time.perf_counter()
        oracle_call(kind, small)
        single = small[0].shape[0] / (time.perf_counter() - t0)
    finally:
        torch.set_num_threads(cores)
    return {"value": sample / mean, "unit": "matrices/s", "cores": torch.get_num_threads(), "kind": reference_impl()[0],
            "cpu_model": cpu_model(), "single_thread_value": single,
            "sample": f"{sample} of {batch} matrices per step, {steps} steps after {warmup} warm-up; " + reference_impl()[2],
            "best_value": sample / min(times), "seconds_per_step": mean, "sample_matrices": sample}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sym_solve3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="override the workload's batch (debug)")
    ap.add_argument("--kind", default=None, help="custom workload: sym_solve|sym_matvec|sym_invert|batch_inv|batch_det|batch_solve")
    ap.add_argument("--n", type=int, default=None, help="custom workload: matrix order")
    ap.add_argument("--dtype", default=None, choices=["f32", "f64"], help="custom workload: scalar type")
    ap.add_argument("--method", default="auto", choices=sorted(ALGOS), help="factorisation for sym_solve / sym_invert, N > 4")
    ap.add_argument("--launch", default=os.environ.get("NFM_BENCH_LAUNCH", "graph"), choices=["graph", "eager"],
                    help="how the K timed steps reach the GPU: 'graph' = the K C-ABI calls captured once in a CUDA graph and "
                         "replayed inside the timed region (the host cannot stall a 16 us launch); 'eager' = K ctypes calls")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--workloads", default=None,
                    help="comma-separated list: several workloads in one process, one JSON line each (saves start-up on multi-GPU boxes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output of the last timed step, shaped as the public API returns it, "
                         "as DIR/<workload>.npy "
                         "(DIR/<workload>.rank<R>.npy per rank when N > 1), in the workload's dtype; outputs above "
                         f"{DUMP_BUDGET >> 20} MiB in all are cut to a fixed, seeded sample of rows (in ascending order)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world != 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    dist = None
    if args.impl == "ours" and world > 1:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU path in the product)")
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    names = args.workloads.split(",") if args.workloads else [args.workload]
    for name in names:
        if name not in WORKLOADS:
            raise SystemExit(f"unknown workload {name}")
        args.workload = name
        run_workload(args, rank, local_rank, world, dist, DUMP_BUDGET // (len(names) * world))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_output(out: torch.Tensor, path: str, budget: int) -> None:
    """Write ``out`` (one record per row) to ``path`` as .npy; above ``budget`` bytes, a
    sample of rows drawn with a fixed seed, so that two runs with the same arguments write
    the same rows."""
    import numpy as np
    rows = out.shape[0]
    keep = max(1, budget // max(1, out[:1].numel() * out.element_size()))
    if rows > keep:
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out = out[idx.to(out.device)]
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    np.save(path, out.cpu().numpy())


def run_workload(args, rank, local_rank, world, dist, dump_budget):

    w = dict(WORKLOADS[args.workload])
    if args.kind or args.n or args.dtype:
        w["kind"] = args.kind or w["kind"]
        w["n"] = args.n or w["n"]
        w["dtype"] = args.dtype or w["dtype"]
        w["batch"] = args.batch or w["batch"]
        w["desc"] = "custom: %s n=%d %s batch=%d" % (w["kind"], w["n"], w["dtype"], w["batch"])
    kind, n = w["kind"], w["n"]
    dtype = torch.float32 if w["dtype"] == "f32" else torch.float64
    esize = 4 if dtype == torch.float32 else 8
    batch = args.batch or w["batch"]
    alg = algorithmic_bytes(kind, n, esize)
    # the same keys and values in both arms (the driver compares them)
    config = {"workload": w["desc"], "routine": kind, "n": n, "batch": batch, "bytes_per_matrix": alg, "method": args.method,
              "l2": "working set per GPU larger than L2, or >= 3x L2 of rotated operand sets (see timing.l2)"}
    timing = {}

    if args.impl == "reference":
        if rank != 0:
            return
        base = cpu_baseline(kind, n, dtype, batch, steps=args.steps, warmup=args.warmup, budget_s=120.0)
        line = {"impl": "reference", "metric": "batched sym-solve matrices/sec" if kind == "sym_solve" else f"{kind} matrices/sec",
                "value": base["value"], "unit": "matrices/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": base["seconds_per_step"] * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": w["dtype"],
                "data": "synthetic", "config": config, "cpu_baseline": base,
                "e2e": {"value": base["value"], "unit": "matrices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path in the product)")
    from nitorch_fastmath_b200 import _lib
    from nitorch_fastmath_b200.shard import shard_bounds
    lib = _lib.load()

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and os.environ.get("NFM_BENCH_BIND") == "1":   # optional: measured no gain on this pool's hosts
        timing["cpu_affinity"] = bind_to_gpu_cpus(local_rank)
    begin, end = shard_bounds(batch, world, rank)
    my = end - begin
    code = 0 if dtype == torch.float32 else 1
    lens, olen = record_lengths(kind, n)

    set_bytes = my * alg
    nsets = operand_set_count(set_bytes)
    sets = []
    for s in range(nsets):
        ins = make_inputs(kind, n, dtype, my, dev, seed=operand_seed(rank, s))
        out = torch.empty(my, olen, device=dev, dtype=dtype) if olen > 1 else torch.empty(my, device=dev, dtype=dtype)
        sets.append((ins, out))
    timing["l2"] = (f"per-GPU working set {set_bytes / 2**20:.0f} MiB > L2" if nsets == 1 else
                    f"rotating {nsets} operand sets of {set_bytes / 2**20:.0f} MiB (> 3x L2 in total)")

    # everything device-resident runs on one side stream (CUDA graphs cannot be captured on the legacy
    # default stream); the timing events are recorded on that same stream
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    torch.cuda.set_stream(side)
    stream = side.cuda_stream
    launchers = [abi_launcher(lib, kind, n, code, my, ins, out, stream, ALGOS[args.method]) for ins, out in sets]

    def step(i):
        rc = launchers[i % nsets]()
        if rc:
            _lib.check(rc, "bench step")

    def sync():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(dev)

    clocks = ClockSampler(local_rank)
    for i in range(args.warmup):
        step(i)
    clocks.wait_ready()
    # the timed loop is as tight as Python allows: pre-bound C-ABI calls, return codes checked afterwards
    seq = [launchers[timed_set(args.warmup, i, nsets)] for i in range(args.steps)]
    sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rc_any = 0
    graph = None
    if args.launch == "graph":
        # the K steps (K calls of the C ABI, one per operand set in rotation) are captured ONCE; the
        # timed region replays them.  Programmatic (PDL) edges between the launches survive capture.
        try:
            graph = torch.cuda.CUDAGraph()
            launches0 = _lib.launch_count()
            with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                for f in seq:
                    rc_any |= f()
            launches = _lib.launch_count() - launches0  # kernel nodes in the graph = launches per replay
            graph.replay()                              # untimed: the first replay uploads the executable graph
        except Exception as exc:                        # e.g. another thread of the process broke the capture
            print("bench.py: CUDA graph capture failed (%s); timing eager launches instead" % exc, file=sys.stderr)
            graph, rc_any = None, 0
            torch.cuda.synchronize(dev)
    if graph is not None:
        if rc_any:
            _lib.check(rc_any, "bench step (capture)")
        sync()
        with clocks:
            ev0.record()
            graph.replay()
            ev1.record()
            sync()
        timing["launch"] = "cuda graph: %d steps captured through the C ABI, one replay timed" % args.steps
    else:
        if args.launch == "graph":
            sync()          # a rank whose capture failed keeps the barrier count of the ranks that replay
        launches0 = _lib.launch_count()
        with clocks:
            ev0.record()
            for f in seq:
                rc_any |= f()
            ev1.record()
            sync()
        if rc_any:
            _lib.check(rc_any, "bench step")
        launches = _lib.launch_count() - launches0
        timing["launch"] = "eager: %d ctypes calls of the C ABI" % args.steps
    if args.dump_outputs:
        last_out = sets[timed_set(args.warmup, args.steps - 1, nsets)][1]
        if kind == "batch_inv":         # the public batchinv returns (..., n, n)
            last_out = last_out.view(my, n, n)
        suffix = ".rank%d" % rank if world > 1 else ""
        dump_output(last_out, os.path.join(args.dump_outputs, args.workload + suffix + ".npy"), dump_budget)
    elapsed_ms = ev0.elapsed_time(ev1)
    if dist is not None:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = batch / (ms_per_step * 1e-3)

    # roofline of the dominant kernel: algorithmic bytes per launch / average launch duration
    peak, peak_src = measured_peak()
    local_ms = ev0.elapsed_time(ev1) / args.steps
    achieved = my * alg / (local_ms * 1e-3) / 1e9
    path = int(lib.nfm_last_path_was_tma())
    kernel = {1: "nfm::tile_kernel", 2: "nfm::warp_solve_kernel", 3: "nfm::pool_kernel", 4: "nfm::solve_many_staged_kernel", 0: "nfm::strided_kernel"}[path]
    # dram bytes per launch come from a committed ncu capture of the default single-GPU run of this
    # workload (profiles/traffic.json): a lookup, not a measurement of this run -- null otherwise
    default_run = world == 1 and args.method == "auto" and batch == WORKLOADS[args.workload]["batch"] and not (args.kind or args.n or args.dtype)
    traffic = recorded_traffic(args.workload) if default_run else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": "profiles/traffic.json (ncu --set full capture of this workload at 1 GPU; not measured in this run)" if traffic else None,
                "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                "kernel": "%s<%s n=%d %s> (%d launch(es) per step per GPU, TMA-staged)" % (kernel, kind, n, w["dtype"], launches // max(args.steps, 1)),
                "bytes_per_launch": my * alg, "avg_launch_us": local_ms * 1e3}

    # small working sets: the same K steps on ONE operand set, i.e. with the data resident in the
    # 126 MB L2 -- reported next to the HBM figure above (rotated sets), never instead of it
    if nsets > 1:
        one = [launchers[0]] * args.steps
        for f in one[:3]:
            f()
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for f in one:
            f()
        e1.record()
        sync()
        l2_ms = e0.elapsed_time(e1) / args.steps
        roofline["l2_resident"] = {"avg_launch_us": l2_ms * 1e3, "achieved": my * alg / (l2_ms * 1e-3) / 1e9, "unit": "GB/s",
                                   "note": "same launches on one operand set (%.0f MiB, stays in L2): NOT an HBM figure" % (set_bytes / 2**20)}

    # end to end: host (pinned) operands through the public API
    e2e = None
    if not args.no_e2e:
        ins0, _ = sets[0]
        # a bounded slab for the 17 GB dense workloads: the e2e rate is set by PCIe, not by the size
        e2e_n = min(my, max(1 << 20, int(2e9) // alg))
        host_in = [t[:e2e_n].cpu().pin_memory() for t in ins0]
        host_out = (torch.empty((e2e_n, olen), dtype=dtype) if olen > 1 else torch.empty((e2e_n,), dtype=dtype)).pin_memory()
        if kind == "batch_inv":
            host_out = host_out.view(e2e_n, n, n)
        ksteps = args.e2e_steps or max(3, min(args.steps, 10))
        for _ in range(2):
            api_call(kind, host_in, host_out)
        sync()
        t0 = time.perf_counter()
        for _ in range(ksteps):
            api_call(kind, host_in, host_out)   # synchronises its pipeline streams before returning
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": e2e_n * world / (dt / ksteps), "unit": "matrices/s",
               "h2d_bytes_per_step": sum(t.numel() * esize for t in host_in) * world,
               "d2h_bytes_per_step": host_out.numel() * esize * world, "steps": ksteps,
               "ms_per_step": dt / ksteps * 1e3, "matrices_per_step": e2e_n * world,
               "api": "nitorch_fastmath_b200 %s(pinned CPU tensors%s)" % (kind, ", out=pinned CPU tensor")}

    base = None
    if rank == 0 and world == 1 and not args.no_cpu:
        base = cpu_baseline(kind, n, dtype, batch, steps=3, warmup=1, budget_s=20.0)

    if rank == 0:
        line = {"metric": "batched sym-solve matrices/sec" if kind == "sym_solve" else f"{kind} matrices/sec",
                "value": value, "unit": "matrices/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": w["dtype"], "data": "synthetic", "config": config, "timing": timing, "roofline": roofline,
                "clocks": clocks.summary(), "gpu_launches": int(launches), "e2e": e2e}
        if base is not None:
            line["cpu_baseline"] = base
        print(json.dumps(line), flush=True)
    del sets, launchers
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
