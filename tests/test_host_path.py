"""CPU operands: the chunked H2D -> kernel -> D2H pipelines (``nfm_*_host``) and every
route by which the public API takes CPU tensors.

The package has no CPU path.  A dense CPU batch is streamed through the GPU by the host
pipelines; anything else is uploaded whole and computed with the device entry point.
Every result is checked twice:

* exact: the same inputs through the device entry point must give the same bits
  (results do not depend on batch size or tile geometry, DESIGN section 4, so cutting
  the batch into chunks must not change a bit).  ``method='warp'`` is the exception:
  each chunk's ragged remainder leaves the sub-warp kernel, so there the device call
  is made on the same chunk cuts;
* accurate: every matrix against a float64 reference of the same operation, at the
  parity tests' bars.

The pipeline itself is driven through the C ABI at chunk sizes from 1 to past the
batch, 1 to 5 buffers (also one stream passed several times), pinned and pageable
buffers and in place, with guard zones around ``h_out`` and behind the workspace.
The argument and workspace checks run without a GPU.
"""
from __future__ import annotations

import ctypes
import hashlib
import json
import math
import os
import subprocess
import sys
import threading

import pytest
import torch

from conftest import ROOT, TOL
from oracle import generators as G
from oracle import ref_port as P
from nitorch_fastmath_b200 import _lib

DEV = "cuda:0"
DTYPES = [torch.float32, torch.float64]
CODE = {torch.float32: _lib.F32, torch.float64: _lib.F64}
ALGO = {"auto": _lib.ALGO_AUTO, "ldl": _lib.ALGO_LDL, "lu": _lib.ALGO_LU, "warp": _lib.ALGO_WARP,
        "chol": _lib.ALGO_LDL}
SENTINEL = -1.25e30        # fills every buffer the code under test must not write
GUARD = 37                 # elements of guard zone on each side of h_out
WS_GUARD = 4096            # bytes of guard behind the device workspace


def _nfm():
    import nitorch_fastmath_b200 as pkg
    return pkg


def _bits(t):
    return t.detach().contiguous().view(-1).view(torch.uint8)


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _pk(n):
    return n * (n + 1) // 2


# --------------------------------------------------------------------------
# float64 references and the error measure
# --------------------------------------------------------------------------

def _full(mat, n):
    """Dense float64 matrix of a packed / diagonal / scaled-identity record."""
    mat = mat.double()
    if mat.shape[-1] == _pk(n):
        return P.sym_to_full(mat)
    if mat.shape[-1] == 1:
        return torch.diag_embed(mat.expand(*mat.shape[:-1], n))
    return torch.diag_embed(mat)


def _solve(a, b):
    return torch.linalg.solve(a, b[..., None])[..., 0]


def worst_err(got, want, rec=1, addend=None):
    """Worst per-matrix norm-wise relative error; for ``inp +/- A v`` relative to |inp| + |A v|."""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    if got.numel() == 0:
        return 0.0
    dims = tuple(range(-rec, 0))
    if rec == 0:
        return float(((got - want).abs() / want.abs().clamp_min(1e-300)).max())
    num = (got - want).pow(2).sum(dims).sqrt()
    if addend is None:
        den = want.pow(2).sum(dims).sqrt()
    else:
        a = addend.cpu().double().expand_as(want)
        den = a.pow(2).sum(dims).sqrt() + (want - a).pow(2).sum(dims).sqrt()
    return float((num / den.clamp_min(1e-300)).max())


def bar(res_dtype, *in_dtypes, scale=1.0):
    """TOL of the precision the call computes in; a half / bfloat16 result adds its own rounding."""
    dts = (res_dtype,) + tuple(in_dtypes)
    tol = TOL[torch.float64 if all(d == torch.float64 for d in dts) else torch.float32] * scale
    if res_dtype in (torch.float16, torch.bfloat16):
        tol = max(tol, torch.finfo(res_dtype).eps)
    return tol


# --------------------------------------------------------------------------
# C ABI: one spec per host entry and operand variant
# --------------------------------------------------------------------------

class Spec:
    """CPU inputs (flat records, None for an absent optional operand), the host entry,
    the device entry on the same records, and a float64 reference."""

    def __init__(self, name, dtype, n, ins, out_rec, host, dev, ref, scale=1.0, addend=None, inplace=None,
                 warp=False):
        self.name, self.dtype, self.n, self.ins, self.out_rec = name, dtype, n, ins, out_rec
        self.host, self.dev, self.ref = host, dev, ref
        self.scale, self.addend, self.inplace, self.warp = scale, addend, inplace, warp
        self.batch = ins[0].shape[0]
        self.in_elems = [t.shape[-1] for t in ins if t is not None]
        self._dev_out = None

    def __repr__(self):
        return f"{self.name}[{self.dtype}, n={self.n}, batch={self.batch}]"


def _mix(b, n, dtype, seed):
    """SPD matrices with every second one symmetric indefinite (the checked LDL^T falls back per lane)."""
    m = G.spd_packed(b, n, dtype, seed)
    m[1::2] = G.sym_indefinite_packed(b, n, dtype, seed + 1)[1::2]
    return m


def solve_spec(dtype, n, batch, algo="auto", diag=False, mix=False, inplace=False, seed=0):
    a, nn = ALGO[algo], _pk(n)
    mat = (_mix if mix else G.spd_packed)(batch, n, dtype, seed)
    vec = G.vectors(batch, n, dtype, seed + 2)
    # small enough (<= ~0.5) that no indefinite matrix (eigenvalues +-[1, 2]) is moved near singular
    reg = G.vectors(batch, n, dtype, seed + 3).abs() * 0.1 + 0.01 if diag else None

    def ref(ins):
        full = _full(ins[0], n)
        if ins[2] is not None:
            full = full + torch.diag_embed(ins[2].double())
        return _solve(full, ins[1].double())
    return Spec(f"solve_{algo}{'_diag' if diag else ''}{'_mix' if mix else ''}{'_inplace' if inplace else ''}",
                dtype, n, [mat, vec, reg], n,
                lambda L, c, B, p, o, *r: L.nfm_sym_solve_host(c, n, a, B, p[0], p[1], p[2], o, *r),
                lambda L, c, B, p, o, s: L.nfm_sym_solve(c, n, _lib.LAYOUT_SYM, a, B, p[0], nn, p[1], n, p[2],
                                                         n if diag else 0, o, n, s),
                ref, scale=(20 if algo == "auto" else 4) if mix else 1.0, inplace=1 if inplace else None,
                warp=algo == "warp")


def matvec_spec(dtype, n, batch, sign=0, inplace=False, seed=0):
    nn = _pk(n)
    mat = G.spd_packed(batch, n, dtype, seed)
    vec = G.vectors(batch, n, dtype, seed + 2)
    inp = G.vectors(batch, n, dtype, seed + 3) if sign else None

    def ref(ins):
        y = (_full(ins[0], n) @ ins[1].double()[..., None])[..., 0]
        return y if ins[2] is None else ins[2].double() + sign * y
    return Spec(f"matvec_sign{sign}{'_inplace' if inplace else ''}", dtype, n, [mat, vec, inp], n,
                lambda L, c, B, p, o, *r: L.nfm_sym_matvec_host(c, n, B, p[0], p[1], p[2], sign, o, *r),
                lambda L, c, B, p, o, s: L.nfm_sym_matvec(c, n, _lib.LAYOUT_SYM, B, p[0], nn, p[1], n, p[2],
                                                          n if sign else 0, sign, o, n, s),
                ref, addend=2 if sign else None, inplace=2 if inplace else None)


def invert_spec(dtype, n, batch, algo="auto", diag_only=0, inplace=False, seed=0):
    a, nn = ALGO[algo], _pk(n)
    no = n if diag_only else nn
    mat = G.spd_packed(batch, n, dtype, seed)

    def ref(ins):
        inv = torch.linalg.inv(_full(ins[0], n))
        return inv.diagonal(0, -1, -2) if diag_only else P.full_to_sym(inv)
    return Spec(f"invert_{algo}_diag{diag_only}{'_inplace' if inplace else ''}", dtype, n, [mat], no,
                lambda L, c, B, p, o, *r: L.nfm_sym_invert_host(c, n, a, diag_only, B, p[0], o, *r),
                lambda L, c, B, p, o, s: L.nfm_sym_invert(c, n, a, diag_only, B, p[0], nn, o, no, s),
                ref, inplace=0 if inplace else None)


def _dense(dtype, n, batch, spd, seed):
    a = G.dense_spd(batch, n, dtype, seed) if spd else G.dense_shifted(batch, n, dtype, seed)
    return a.reshape(batch, n * n).contiguous()


def batch_inv_spec(dtype, n, batch, algo="auto", reg=0, seed=0):
    a, nn = ALGO[algo], n * n
    return Spec(f"batch_inv_{algo}_reg{reg}", dtype, n, [_dense(dtype, n, batch, algo == "chol", seed)], nn,
                lambda L, c, B, p, o, *r: L.nfm_batch_inv_host(c, n, a, reg, B, p[0], o, *r),
                lambda L, c, B, p, o, s: L.nfm_batch_inv(c, n, a, reg, B, p[0], nn, o, nn, s),
                lambda ins: torch.linalg.inv(ins[0].double().view(-1, n, n)).reshape(-1, nn))


def batch_det_spec(dtype, n, batch, seed=0):
    nn = n * n
    return Spec("batch_det", dtype, n, [_dense(dtype, n, batch, False, seed)], 1,
                lambda L, c, B, p, o, *r: L.nfm_batch_det_host(c, n, B, p[0], o, *r),
                lambda L, c, B, p, o, s: L.nfm_batch_det(c, n, B, p[0], nn, o, 1, s),
                lambda ins: torch.linalg.det(ins[0].double().view(-1, n, n))[:, None])


def batch_solve_spec(dtype, n, batch, nrhs=1, algo="lu", seed=0):
    a, nn, nk = ALGO[algo], n * n, n * nrhs
    b = G.vectors((batch, n), nrhs, dtype, seed + 2).reshape(batch, nk)
    return Spec(f"batch_solve_{algo}_k{nrhs}", dtype, n, [_dense(dtype, n, batch, algo == "chol", seed), b], nk,
                lambda L, c, B, p, o, *r: L.nfm_batch_solve_host(c, n, nrhs, a, B, p[0], p[1], o, *r),
                lambda L, c, B, p, o, s: L.nfm_batch_solve(c, n, nrhs, a, B, p[0], nn, p[1], nk, o, nk, s),
                lambda ins: torch.linalg.solve(ins[0].double().view(-1, n, n),
                                               ins[1].double().view(-1, n, nrhs)).reshape(-1, nk))


def device_result(spec, cuts=None):
    """The device entry on the same records: one call, or one call per chunk of ``cuts`` matrices,
    each on its own 256-byte-aligned copy like a pipeline slot."""
    lib, code, B = _lib.load(), CODE[spec.dtype], spec.batch
    ins = [None if t is None else t.to(DEV) for t in spec.ins]
    out = torch.empty(B, spec.out_rec, dtype=spec.dtype, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream
    for b in range(0, B, cuts or max(B, 1)):
        e = min(B, b + (cuts or B))
        part = [None if t is None else t[b:e].clone() for t in ins]
        o = torch.empty(e - b, spec.out_rec, dtype=spec.dtype, device=DEV)
        _lib.check(spec.dev(lib, code, e - b, [None if t is None else t.data_ptr() for t in part], o.data_ptr(),
                            stream), spec.name)
        out[b:e] = o
    return out.cpu()


def exact_and_accurate(spec, got, chunk):
    """``got`` must equal the device call bit for bit, and every matrix must meet the float64 bar."""
    if spec.warp:
        want = device_result(spec, chunk)
        assert worst_err(got, spec.ref(spec.ins)) <= TOL[spec.dtype] * spec.scale, spec
    else:
        if spec._dev_out is None:
            spec._dev_out = device_result(spec)
            # the device result is checked once; every host result must then equal it bit for bit
            addend = spec.ins[spec.addend] if spec.addend is not None else None
            err = worst_err(spec._dev_out, spec.ref(spec.ins), addend=addend)
            assert err <= TOL[spec.dtype] * spec.scale, f"{spec}: worst rel err {err:.3e}"
        want = spec._dev_out
    assert torch.equal(got, want), f"{spec}, chunk {chunk}: the host pipeline differs from the device call"


def run_pipeline(spec, chunk, nbuf, same_stream=False, pin_in=True, pin_out=True, expect_rc=0):
    """One call of the host entry with guard zones around h_out and behind the workspace.
    With ``expect_rc`` set, the call must fail with that code and leave h_out untouched."""
    lib, code, B = _lib.load(), CODE[spec.dtype], spec.batch
    dummy = torch.zeros(16, dtype=spec.dtype)      # an empty batch still passes non-NULL pointers
    ins = [None if t is None else (t.pin_memory() if pin_in else t.clone()) for t in spec.ins]
    numel = B * spec.out_rec
    buf = torch.full((numel + 2 * GUARD,), SENTINEL, dtype=spec.dtype)
    if pin_out:
        buf = buf.pin_memory()
    out = buf[GUARD:GUARD + numel].view(B, spec.out_rec)
    if spec.inplace is not None:
        out.copy_(spec.ins[spec.inplace])
        ins[spec.inplace] = out
    before = buf.clone()
    ws_bytes = int(lib.nfm_host_workspace_bytes(code, chunk, nbuf, sum(spec.in_elems), spec.out_rec))
    ws = torch.full((ws_bytes + WS_GUARD,), 0xA5, dtype=torch.uint8, device=DEV)
    streams = ([torch.cuda.Stream(device=DEV)] * nbuf if same_stream else
               [torch.cuda.Stream(device=DEV) for _ in range(nbuf)])
    arr = (ctypes.c_void_p * nbuf)(*[s.cuda_stream for s in streams])
    torch.cuda.synchronize()                       # the workspace fill must land before the pipeline streams run
    launches = _lib.launch_count()
    rc = spec.host(lib, code, B, [None if t is None else (t.data_ptr() if B else dummy.data_ptr()) for t in ins],
                   out.data_ptr() if B else dummy.data_ptr(), ws.data_ptr(), ws_bytes, chunk, nbuf, arr)
    launches = _lib.launch_count() - launches
    if expect_rc:
        assert rc == expect_rc and same_bits(buf, before), (spec, rc)
        return None
    _lib.check(rc, spec.name)
    assert launches >= -(-B // chunk), (spec, chunk, launches)       # the pipeline really cut the batch
    assert same_bits(buf[:GUARD], before[:GUARD]) and same_bits(buf[GUARD + numel:], before[GUARD + numel:]), \
        f"{spec}: write outside h_out"
    assert bool((ws[ws_bytes:] == 0xA5).all()), f"{spec}: write past the workspace"
    for i, (t, orig) in enumerate(zip(ins, spec.ins)):
        if t is not None and i != spec.inplace:
            assert same_bits(t, orig), f"{spec}: input {i} changed"
    if B == 0:
        assert same_bits(buf, before) and launches == 0
    return out.clone()


def grid_specs(dtype, n, batch):
    return [solve_spec(dtype, n, batch, "auto", diag=True, mix=True),
            solve_spec(dtype, n, batch, "ldl", inplace=True, seed=1),
            matvec_spec(dtype, n, batch, sign=-1),
            matvec_spec(dtype, n, batch, sign=+1, inplace=True, seed=1),
            invert_spec(dtype, n, batch, "lu", inplace=True),
            invert_spec(dtype, n, batch, "auto", diag_only=1, seed=1),
            batch_inv_spec(dtype, n, batch, "auto", reg=1),
            batch_det_spec(dtype, n, batch),
            batch_solve_spec(dtype, n, batch, nrhs=5)]


GRID_CHUNKS = [1, 3, 4, 31, 32, 33, 1000, 1024, "batch", "batch+5"]
GRID_NBUF = [(1, False), (2, False), (3, False), (5, False), (2, True), (5, True)]
GRID_ORDERS = [(3, torch.float32), (6, torch.float64), (10, torch.float32)]


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", GRID_CHUNKS, ids=str)
def test_pipeline_chunk_and_ring_grid(chunk):
    """Every entry (solve, in-place solve, matvec and in-place addmatvec, in-place invert, diagonal
    invert, dense inverse, det, 5-column solve) at every chunk size x buffer count; the batch
    gives 16 chunks, so a ring of 5 slots wraps three times, with a ragged last chunk."""
    if chunk == "batch":
        batch, c = 777, 777
    elif chunk == "batch+5":
        batch, c = 777, 782
    else:
        batch, c = 15 * chunk + chunk // 2 + 1, chunk
    for n, dtype in GRID_ORDERS:
        for spec in grid_specs(dtype, n, batch):
            for nbuf, same in GRID_NBUF:
                exact_and_accurate(spec, run_pipeline(spec, c, nbuf, same), c)


PIN_MODES = [(True, True), (False, False), (True, False), (False, True)]


def order_specs(dtype, n, batch):
    specs = []
    for algo in ("auto", "ldl", "lu", "warp"):
        for diag in (False, True):
            specs.append(solve_spec(dtype, n, batch, algo, diag=diag))
    specs += [solve_spec(dtype, n, batch, "auto", mix=True, seed=3), solve_spec(dtype, n, batch, "lu", mix=True, seed=3),
              solve_spec(dtype, n, batch, "auto", diag=True, inplace=True, seed=4)]
    specs += [matvec_spec(dtype, n, batch, s) for s in (0, 1, -1)] + [matvec_spec(dtype, n, batch, -1, inplace=True)]
    specs += [invert_spec(dtype, n, batch, a, d) for a in ("auto", "lu") for d in (0, 1)]
    specs += [invert_spec(dtype, n, batch, "auto", inplace=True, seed=2)]
    specs += [batch_inv_spec(dtype, n, batch, a, r) for a, r in (("auto", 0), ("auto", 1), ("lu", 0), ("chol", 0))]
    specs += [batch_det_spec(dtype, n, batch)]
    specs += [batch_solve_spec(dtype, n, batch, k, a) for k in (1, 2, 3, 4, 5, 8) for a in ("lu", "chol")]
    return specs


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("n", range(1, 11))
def test_every_order_and_operand_variant(n, dtype):
    """Orders 1-10: every algorithm, regulariser, sign, diag_only, closed-form shift and
    right-hand-side count (5 and 8 run the staged many-right-hand-side kernel in each chunk)
    through 1024-matrix chunks on 3 buffers (8 chunks, the ring wraps twice), host buffers
    pinned and pageable in both directions."""
    batch = 7 * 1024 + 333
    for i, spec in enumerate(order_specs(dtype, n, batch)):
        pin_in, pin_out = PIN_MODES[i % 4]
        exact_and_accurate(spec, run_pipeline(spec, 1024, 3, pin_in=pin_in, pin_out=pin_out), 1024)


def edge_specs(batch):
    out = []
    for n, dtype in ((3, torch.float32), (7, torch.float64)):
        out += [solve_spec(dtype, n, batch, diag=True), matvec_spec(dtype, n, batch, 1), invert_spec(dtype, n, batch),
                batch_inv_spec(dtype, n, batch), batch_det_spec(dtype, n, batch), batch_solve_spec(dtype, n, batch, 8)]
    return out


@pytest.mark.gpu
def test_empty_and_single_matrix_batches():
    """batch 0 returns NFM_OK, launches nothing and writes nothing; batch 1 in chunks of 1 and 4."""
    for spec in edge_specs(0):
        run_pipeline(spec, 4, 3)
    for spec in edge_specs(1):
        for chunk in (1, 4):
            exact_and_accurate(spec, run_pipeline(spec, chunk, 3), chunk)


@pytest.mark.gpu
def test_matvec_with_an_addend_and_no_sign_is_rejected_and_writes_nothing():
    spec = matvec_spec(torch.float32, 3, 100, sign=1)
    spec.host = lambda L, c, B, p, o, *r: L.nfm_sym_matvec_host(c, 3, B, p[0], p[1], p[2], 0, o, *r)
    run_pipeline(spec, 32, 3, expect_rc=-2)
    assert b"sign" in _lib.load().nfm_last_error_string()


# --------------------------------------------------------------------------
# argument and workspace checks: all return before any CUDA call
# --------------------------------------------------------------------------

def _need(dtype_code, chunk, nbuf, in_elems, out_elems):
    """Workspace the pipeline uses: each operand chunk and the output chunk 256-byte aligned, per buffer."""
    es = 8 if dtype_code == _lib.F64 else 4
    up = lambda x: -(-x // 256) * 256    # noqa: E731
    return nbuf * (sum(up(chunk * e * es) for e in in_elems) + up(chunk * out_elems * es))


def _abi_calls(n=3, nrhs=2):
    """entry -> (call(n, batch, ins, out, ws, wsb, chunk, nbuf, streams), input records, output record)."""
    nn, sq = _pk(n), n * n
    return {
        "sym_solve": (lambda n, B, i, o, *r: _lib.load().nfm_sym_solve_host(_lib.F32, n, 0, B, i[0], i[1], i[2], o, *r),
                      [nn, n, n], n),
        "sym_invert": (lambda n, B, i, o, *r: _lib.load().nfm_sym_invert_host(_lib.F32, n, 0, 1, B, i[0], o, *r),
                       [nn], n),
        "sym_matvec": (lambda n, B, i, o, *r: _lib.load().nfm_sym_matvec_host(_lib.F32, n, B, i[0], i[1], i[2], 1, o, *r),
                       [nn, n, n], n),
        "batch_inv": (lambda n, B, i, o, *r: _lib.load().nfm_batch_inv_host(_lib.F32, n, 0, 1, B, i[0], o, *r),
                      [sq], sq),
        "batch_det": (lambda n, B, i, o, *r: _lib.load().nfm_batch_det_host(_lib.F32, n, B, i[0], o, *r), [sq], 1),
        "batch_solve": (lambda n, B, i, o, *r: _lib.load().nfm_batch_solve_host(_lib.F32, n, nrhs, 2, B, i[0], i[1], o, *r),
                        [sq, n * nrhs], n * nrhs),
    }


REQUIRED = {"sym_solve": (0, 1), "sym_invert": (0,), "sym_matvec": (0, 1), "batch_inv": (0,), "batch_det": (0,),
            "batch_solve": (0, 1)}


@pytest.mark.parametrize("entry", sorted(REQUIRED))
def test_host_entries_reject_bad_arguments_without_a_gpu(entry):
    """NFM_E_BADARG for chunk < 1, nbuf < 1, a negative batch, NULL streams / workspace / h_out /
    required input and n outside 1-10; NFM_E_WORKSPACE for a workspace one byte short of what
    the pipeline uses (which nfm_host_workspace_bytes bounds), with h_out untouched."""
    lib = _lib.load()
    inbuf = ctypes.create_string_buffer(1 << 16)
    outbuf = ctypes.create_string_buffer(b"\x5a" * (1 << 16), 1 << 16)
    hp, ho = ctypes.addressof(inbuf), ctypes.addressof(outbuf)
    call, in_elems, out_elems = _abi_calls()[entry]
    streams = (ctypes.c_void_p * 3)()
    n, B, chunk, nbuf = 3, 100, 7, 3
    ins = [hp] * 3
    need = _need(_lib.F32, chunk, nbuf, in_elems, out_elems)
    assert need <= lib.nfm_host_workspace_bytes(_lib.F32, chunk, nbuf, sum(in_elems), out_elems)
    ok = dict(n=n, B=B, i=ins, o=ho, ws=hp, wsb=need, chunk=chunk, nbuf=nbuf, streams=streams)

    def rc(**kw):
        a = dict(ok, **kw)
        return call(a["n"], a["B"], a["i"], a["o"], a["ws"], a["wsb"], a["chunk"], a["nbuf"], a["streams"])

    for kw in (dict(chunk=0), dict(chunk=-1), dict(nbuf=0), dict(nbuf=-2), dict(B=-1), dict(streams=None),
               dict(ws=None), dict(o=None), dict(n=0), dict(n=11)):
        assert rc(**kw) == -2, (entry, kw)
    for k in REQUIRED[entry]:
        bad = list(ins)
        bad[k] = None
        assert rc(i=bad) == -2, (entry, k)
    if entry == "batch_solve":
        assert _abi_calls(nrhs=0)[entry][0](n, B, ins, ho, hp, need, chunk, nbuf, streams) == -2
    assert rc(wsb=need - 1) == -3
    assert b"workspace" in lib.nfm_last_error_string()
    assert outbuf.raw == b"\x5a" * (1 << 16)


def test_workspace_bound_covers_the_pipeline_layout():
    """nfm_host_workspace_bytes (one total of the input records) bounds the per-operand aligned
    layout for every split of the inputs, chunk size and buffer count the tests use."""
    lib = _lib.load()
    for code in (_lib.F32, _lib.F64):
        for chunk in (1, 3, 4, 31, 32, 33, 1000, 1024, 782, 21504):
            for nbuf in (1, 2, 3, 5):
                for ins, out in (([55, 10, 10], 10), ([6, 3], 3), ([100, 80], 80), ([1], 1), ([16], 1), ([21], 6)):
                    assert _need(code, chunk, nbuf, ins, out) <= lib.nfm_host_workspace_bytes(code, chunk, nbuf,
                                                                                             sum(ins), out)


# --------------------------------------------------------------------------
# public API with CPU tensors
# --------------------------------------------------------------------------

API_ORDERS = [(1, torch.float64), (3, torch.float32), (6, torch.float64), (10, torch.float32)]
API_B = 2053


def _to_dev(x):
    return x.to(DEV) if torch.is_tensor(x) else x


def _place(t, pinned):
    return t.pin_memory() if pinned else t.clone()


def check_route(fn, args, kw=None, ref=None, tol=None, rec=1, addend=None, pinned=True, out_dtype=None):
    """``fn`` on CPU tensors against ``fn`` on the same tensors moved to the GPU: shape, dtype,
    device and bits; then the float64 reference; then ``out=`` (written in place, pointer kept)."""
    kw = kw or {}
    before = [a.clone() for a in args if torch.is_tensor(a)]
    got = fn(*args, **kw)
    want = fn(*[_to_dev(a) for a in args], **{k: _to_dev(v) for k, v in kw.items()})
    assert got.device.type == "cpu"
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, want.shape, got.dtype, want.dtype)
    assert torch.equal(got, want.cpu())
    if ref is not None:
        err = worst_err(got, ref, rec, addend)
        assert err <= tol, f"rel err {err:.3e} > {tol:.1e}"
    for a, b in zip([a for a in args if torch.is_tensor(a)], before):
        assert same_bits(a, b)
    odt = out_dtype or got.dtype
    out = torch.full(got.shape, SENTINEL, dtype=odt) if odt.is_floating_point and odt.itemsize >= 4 else \
        torch.zeros(got.shape, dtype=odt)
    out = _place(out, pinned)
    dout = torch.zeros(got.shape, dtype=odt, device=DEV)
    r = fn(*args, **kw, out=out)
    fn(*[_to_dev(a) for a in args], **{k: _to_dev(v) for k, v in kw.items()}, out=dout)
    assert r.data_ptr() == out.data_ptr() and r.shape == got.shape
    assert torch.equal(out, dout.cpu())
    if out_dtype is None:
        assert torch.equal(out, got)
    return got


def check_inplace(fn, args, target, kw=None):
    """In-place variant on CPU tensors: returns ``args[target]`` itself, with the CUDA call's bits."""
    kw = kw or {}
    dargs = [_to_dev(a) for a in args]
    ptr = args[target].data_ptr()
    r = fn(*args, **kw)
    fn(*dargs, **kw)
    assert r.data_ptr() == ptr and r.device.type == "cpu"
    assert torch.equal(args[target], dargs[target].cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
@pytest.mark.parametrize("n,dtype", API_ORDERS, ids=[f"n{n}_{str(d)[-7:]}" for n, d in API_ORDERS])
def test_api_sym_streamed_routes(n, dtype, pinned):
    """Dense packed CPU batches go through the host pipelines: matvec / addmatvec / submatvec,
    solve (no regulariser, per-voxel field; auto / lu / ldl / warp), invert (full and diagonal,
    auto / lu), the in-place variants; det / to_full / outer / matmul are uploaded whole."""
    nfm = _nfm()
    B, nn = API_B, _pk(n)
    mat = _place(G.spd_packed(B, n, dtype, 1), pinned)
    vec, inp = _place(G.vectors(B, n, dtype, 2), pinned), _place(G.vectors(B, n, dtype, 3), pinned)
    reg = _place(G.vectors(B, n, dtype, 4).abs() + 0.1, pinned)
    A = _full(mat, n)
    Av = (A @ vec.double()[..., None])[..., 0]
    t = bar(dtype)
    check_route(nfm.sym_matvec, (mat, vec), ref=Av, tol=t, pinned=pinned)
    check_route(nfm.sym_addmatvec, (inp, mat, vec), ref=inp.double() + Av, addend=inp, tol=t, pinned=pinned)
    check_route(nfm.sym_submatvec, (inp, mat, vec), ref=inp.double() - Av, addend=inp, tol=t, pinned=pinned)
    for method in (None, "lu", "ldl", "warp"):
        check_route(nfm.sym_solve, (mat, vec), dict(method=method), ref=_solve(A, vec.double()), tol=t, pinned=pinned)
    check_route(nfm.sym_solve, (mat, vec, reg), ref=_solve(A + torch.diag_embed(reg.double()), vec.double()), tol=t,
                pinned=pinned)
    inv = torch.linalg.inv(A)
    for method in (None, "lu"):
        check_route(nfm.sym_invert, (mat,), dict(method=method), ref=P.full_to_sym(inv), tol=t, pinned=pinned)
        check_route(nfm.sym_invert, (mat, True), dict(method=method), ref=inv.diagonal(0, -1, -2), tol=t,
                    pinned=pinned)
    check_inplace(nfm.sym_addmatvec_, [inp.clone(), mat, vec], 0)
    check_inplace(nfm.sym_submatvec_, [inp.clone(), mat, vec], 0)
    check_inplace(nfm.sym_solve_, [mat, vec.clone()], 1)
    check_inplace(nfm.sym_solve_, [mat, vec.clone(), reg], 1, dict(method="lu"))
    check_inplace(nfm.sym_invert_, [mat.clone()], 0)
    # whole-upload functions (no out=)
    for fn, args, ref, rec, scale in ((nfm.sym_det, (mat,), torch.linalg.det(A), 0, 10),
                                      (nfm.sym_to_full, (mat,), A, 2, 1),
                                      (nfm.sym_outer, (vec,), P.sym_outer(vec.double()), 1, 1)):
        got = fn(*args)
        want = fn(*[a.to(DEV) for a in args])
        assert got.device.type == "cpu" and got.shape == want.shape and got.dtype == want.dtype
        assert torch.equal(got, want.cpu())
        assert worst_err(got, ref, rec) <= t * scale
    d = 3 if n != 3 else 2
    j = _place(G.vectors((B, n), d, dtype, 5), pinned)
    got = nfm.sym_matmul(j, mat)
    assert got.device.type == "cpu" and torch.equal(got, nfm.sym_matmul(j.to(DEV), mat.to(DEV)).cpu())
    jd = j.double()
    assert worst_err(got, P.full_to_sym(jd.transpose(-1, -2) @ A @ jd)) <= t


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype", API_ORDERS, ids=[f"n{n}_{str(d)[-7:]}" for n, d in API_ORDERS])
def test_api_sym_uploaded_routes(n, dtype):
    """Every reason to leave the streamed route: diagonal and scaled-identity layouts, partially
    broadcast operands, non-contiguous views, half / bfloat16, mixed dtypes, scalar / sequence /
    1-D regularisers, an out= of another dtype; plus empty and unbatched inputs."""
    nfm = _nfm()
    B, nn = API_B, _pk(n)
    other = torch.float32 if dtype == torch.float64 else torch.float64
    mat = G.spd_packed(B, n, dtype, 1).pin_memory()
    vec, inp = G.vectors(B, n, dtype, 2).pin_memory(), G.vectors(B, n, dtype, 3)
    dg, sc = G.vectors(B, n, dtype, 6).abs() + 0.5, G.vectors(B, 1, dtype, 7).abs() + 0.5
    A = _full(mat, n)
    t = bar(dtype)

    def solve_ref(m, v, r=None):
        full = _full(m, n)
        if r is not None:
            full = full + torch.diag_embed(torch.as_tensor(r, dtype=torch.float64).expand(*full.shape[:-1]))
        return _solve(full, v.double())

    def mv_ref(m, v):
        return (_full(m, n) @ v.double()[..., None])[..., 0]

    # diagonal / scaled-identity layouts
    for m in (dg, sc):
        check_route(nfm.sym_matvec, (m, vec), ref=mv_ref(m, vec), tol=t)
        check_route(nfm.sym_addmatvec, (inp, m, vec), ref=inp.double() + mv_ref(m, vec), addend=inp, tol=t)
        check_route(nfm.sym_solve, (m, vec), ref=solve_ref(m, vec), tol=t)
        check_route(nfm.sym_solve, (m, vec, 0.5), ref=solve_ref(m, vec, 0.5), tol=t)
    # partially broadcast operands: one field of matrices for two right-hand-side fields
    v2 = G.vectors((2, B), n, dtype, 8)
    check_route(nfm.sym_solve, (mat, v2), ref=solve_ref(mat, v2), tol=t)
    check_route(nfm.sym_matvec, (mat, v2), ref=mv_ref(mat, v2), tol=t)
    check_route(nfm.sym_submatvec, (inp, mat, v2), ref=inp.double() - mv_ref(mat, v2), addend=inp.expand(2, B, n),
                tol=t)
    # non-contiguous views
    wide = torch.zeros(B, 2 * nn, dtype=dtype)
    wide[:, ::2] = mat
    mat_nc = wide[:, ::2]
    vec_nc = vec.t().contiguous().t()
    check_route(nfm.sym_solve, (mat_nc, vec_nc), ref=solve_ref(mat, vec), tol=t)
    check_route(nfm.sym_matvec, (mat_nc, vec), ref=mv_ref(mat, vec), tol=t)
    check_route(nfm.sym_invert, (mat_nc,), ref=P.full_to_sym(torch.linalg.inv(A)), tol=t)
    check_route(nfm.sym_invert, (mat_nc, True), dict(method="lu"), ref=torch.linalg.inv(A).diagonal(0, -1, -2), tol=t)
    # regularisers that are not a per-voxel field
    check_route(nfm.sym_solve, (mat, vec, 0.25), ref=solve_ref(mat, vec, 0.25), tol=t)
    seq = [0.5, 0.25][:n]
    check_route(nfm.sym_solve, (mat, vec, seq), ref=solve_ref(mat, vec, seq + [seq[-1]] * (n - len(seq))), tol=t)
    r1 = G.vectors(1, n, dtype, 9)[0].abs() + 0.1
    check_route(nfm.sym_solve, (mat, vec, r1), ref=solve_ref(mat, vec, r1.double()), tol=t)
    check_route(nfm.sym_solve, (mat, vec), dict(eps=0.5), ref=solve_ref(mat, vec, 0.5), tol=t)
    # half / bfloat16 inputs (computed in float32, returned in the input dtype)
    for low in (torch.float16, torch.bfloat16):
        ml, vl = mat.to(low), vec.to(low)
        check_route(nfm.sym_solve, (ml, vl), ref=solve_ref(ml, vl), tol=bar(low))
        check_route(nfm.sym_matvec, (ml, vl), ref=mv_ref(ml, vl), tol=bar(low))
        check_route(nfm.sym_invert, (ml,), ref=P.full_to_sym(torch.linalg.inv(_full(ml, n))), tol=bar(low))
    # mixed dtypes
    vo = vec.to(other)
    check_route(nfm.sym_solve, (mat, vo), ref=solve_ref(mat, vo), tol=bar(other, dtype))
    check_route(nfm.sym_matvec, (mat, vo), ref=mv_ref(mat, vo), tol=bar(torch.float64, dtype, other))
    check_route(nfm.sym_solve, (mat, vec, G.vectors(B, n, other, 4).abs() + 0.1))
    # an out= of another dtype
    check_route(nfm.sym_solve, (mat, vec), out_dtype=other)
    check_route(nfm.sym_matvec, (mat, vec), out_dtype=other)
    check_route(nfm.sym_invert, (mat,), out_dtype=other)
    check_route(nfm.sym_invert, (mat, True), out_dtype=other)
    # empty and unbatched
    for args in ((mat[:0], vec[:0]), (mat[0], vec[0]), (mat[:1], vec[:1])):
        check_route(nfm.sym_solve, args, ref=solve_ref(*args), tol=t)
        check_route(nfm.sym_matvec, args, ref=mv_ref(*args), tol=t)
        check_route(nfm.sym_invert, args[:1], ref=P.full_to_sym(torch.linalg.inv(_full(args[0], n))), tol=t)
        check_route(nfm.sym_invert, (args[0], True), ref=torch.linalg.inv(_full(args[0], n)).diagonal(0, -1, -2), tol=t)
    check_route(nfm.sym_addmatvec, (inp[0], mat[0], vec[0]), ref=inp[0].double() + mv_ref(mat[0], vec[0]),
                addend=inp[0], tol=t)
    for fn in (nfm.sym_det, nfm.sym_to_full):
        for m in (mat[:0], mat[0]):
            assert torch.equal(fn(m), fn(m.to(DEV)).cpu()) and fn(m).device.type == "cpu"
    assert torch.equal(nfm.sym_outer(vec[0]), nfm.sym_outer(vec[0].to(DEV)).cpu())


DENSE_ORDERS = [(1, torch.float64), (3, torch.float32), (4, torch.float64), (7, torch.float32), (10, torch.float64)]


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
@pytest.mark.parametrize("n,dtype", DENSE_ORDERS, ids=[f"n{n}_{str(d)[-7:]}" for n, d in DENSE_ORDERS])
def test_api_dense_routes(n, dtype, pinned):
    """batchinv / batchdet / batchmatvec / lmdiv / rmdiv / inv / solvevec with lu and chol, on
    the streamed route and on every reason to upload whole."""
    nfm = _nfm()
    B = API_B
    other = torch.float32 if dtype == torch.float64 else torch.float64
    a = _place(G.dense_shifted(B, n, dtype, 1), pinned)
    s = _place(G.dense_spd(B, n, dtype, 2), pinned)
    b = _place(G.vectors(B, n, dtype, 3), pinned)
    ad, sd = a.double(), s.double()
    t = bar(dtype)
    for method, m, md in (("auto", a, ad), ("lu", a, ad), ("chol", s, sd)):
        check_route(nfm.batchinv, (m,), dict(method=method), ref=torch.linalg.inv(md), rec=2, tol=t, pinned=pinned)
    check_route(nfm.batchinv, (a,), dict(regularise=False), ref=torch.linalg.inv(ad), rec=2, tol=t, pinned=pinned)
    check_route(nfm.batchdet, (a,), ref=torch.linalg.det(ad), rec=0, tol=t, pinned=pinned)
    check_route(nfm.batchmatvec, (a, b), ref=(ad @ b.double()[..., None])[..., 0], tol=t, pinned=pinned)
    for method, m, md in (("lu", a, ad), ("chol", s, sd)):
        check_route(nfm.inv, (m, method), ref=torch.linalg.inv(md), rec=2, tol=t, pinned=pinned)
        check_route(nfm.solvevec, (m, b, method), ref=_solve(md, b.double()), tol=t, pinned=pinned)
        for k in (1, 3, 5, 8):
            rhs = _place(G.vectors((B, n), k, dtype, 10 + k), pinned)
            check_route(nfm.lmdiv, (m, rhs, method), ref=torch.linalg.solve(md, rhs.double()), rec=2, tol=t,
                        pinned=pinned)
            lhs = rhs.transpose(-1, -2).contiguous()
            check_route(nfm.rmdiv, (lhs, m, method), ref=lhs.double() @ torch.linalg.inv(md), rec=2, tol=t,
                        pinned=pinned)
    if not pinned:
        return
    # reasons to upload whole
    a_nc = a.transpose(-1, -2).contiguous().transpose(-1, -2)       # the same matrices, column-major records
    check_route(nfm.batchinv, (a_nc,), ref=torch.linalg.inv(ad), rec=2, tol=t)
    check_route(nfm.batchdet, (a[::2],), ref=torch.linalg.det(ad[::2]), rec=0, tol=t)
    check_route(nfm.solvevec, (a_nc, b), ref=_solve(ad, b.double()), tol=t)
    rhs = G.vectors((B, n), 3, dtype, 20)
    check_route(nfm.lmdiv, (a, rhs.to(other)), ref=torch.linalg.solve(ad, rhs.double()), rec=2, tol=bar(other, dtype))
    r2 = G.vectors((2, B, n), 3, dtype, 21)
    check_route(nfm.lmdiv, (a, r2), ref=torch.linalg.solve(ad, r2.double()), rec=2, tol=t)
    check_route(nfm.batchmatvec, (a, G.vectors((2, B), n, dtype, 22)))
    for low in (torch.float16, torch.bfloat16):
        check_route(nfm.batchinv, (a.to(low),), ref=torch.linalg.inv(a.to(low).double()), rec=2, tol=bar(torch.float32))
    check_route(nfm.batchinv, (a,), out_dtype=other)
    check_route(nfm.batchdet, (a,), out_dtype=other)
    check_route(nfm.lmdiv, (a, rhs), out_dtype=other)
    for args in ((a[:0],), (a[0],), (a[:1],)):
        check_route(nfm.batchinv, args, ref=torch.linalg.inv(args[0].double()), rec=2, tol=t)
        check_route(nfm.batchdet, args, ref=torch.linalg.det(args[0].double()), rec=0, tol=t)
        check_route(nfm.lmdiv, (args[0], rhs[:args[0].shape[0]] if args[0].dim() == 3 else rhs[0]))
        check_route(nfm.solvevec, (args[0], b[:args[0].shape[0]] if args[0].dim() == 3 else b[0]))


# --------------------------------------------------------------------------
# out= of the wrong shape: rejected on every CPU route before anything is copied
# --------------------------------------------------------------------------

def _wrong_outs(shape, dtype):
    """Mis-shaped outs, each a view at the start of a sentinel buffer with room for twice the
    result, so that even code that ignored the shape would write inside the buffer."""
    shape = tuple(shape)
    cands = [(*shape[:-1], shape[-1] + 1), (2, *shape)]
    if shape and shape[0] > 1:
        cands += [(shape[0] - 1, *shape[1:]), (shape[0] + 1, *shape[1:])]
    if len(shape) >= 2 and shape[-1] > 1:
        cands.append((*shape[:-1], shape[-1] - 1))
    for ws in cands:
        buf = torch.full((2 * math.prod(shape) + 64,), SENTINEL, dtype=dtype).pin_memory()
        yield buf, buf[:math.prod(ws)].view(ws)


def _rejects(fn, args, kw, shape, dtype):
    before = [a.clone() for a in args if torch.is_tensor(a)]
    for buf, out in _wrong_outs(shape, dtype):
        ref = buf.clone()
        launches = _lib.launch_count()
        with pytest.raises(RuntimeError, match="out has shape"):
            fn(*args, **kw, out=out)
        assert same_bits(buf, ref), f"out {tuple(out.shape)} was written"
        assert _lib.launch_count() == launches, "a rejected call launched work"
    for a, b in zip([a for a in args if torch.is_tensor(a)], before):
        assert same_bits(a, b)


@pytest.mark.gpu
def test_wrong_layout_out_is_rejected():
    """sym_invert(diag=True) of CPU operands with an out of the full packed width: the streamed
    route used to pack B x N values into the head of that buffer and return it."""
    nfm = _nfm()
    B, n = 1000, 4
    mat = G.spd_packed(B, n, torch.float32, 1).pin_memory()
    out = torch.full((B, _pk(n)), SENTINEL).pin_memory()
    ref = out.clone()
    with pytest.raises(RuntimeError, match="out has shape"):
        nfm.sym_invert(mat, True, out=out)
    assert same_bits(out, ref)


def _out_routes(n, dtype):
    nfm = _nfm()
    B, nn = 301, _pk(n)
    mat = G.spd_packed(B, n, dtype, 1).pin_memory()
    vec, inp = G.vectors(B, n, dtype, 2).pin_memory(), G.vectors(B, n, dtype, 3).pin_memory()
    a = G.dense_shifted(B, n, dtype, 4).pin_memory()
    rhs = G.vectors((B, n), 3, dtype, 5).pin_memory()
    half = mat.half()
    return [
        ("sym_matvec streamed", nfm.sym_matvec, (mat, vec), {}, (B, n)),
        ("sym_matvec diagonal", nfm.sym_matvec, (vec.abs() + 1, vec), {}, (B, n)),
        ("sym_addmatvec streamed", nfm.sym_addmatvec, (inp, mat, vec), {}, (B, n)),
        ("sym_submatvec strided", nfm.sym_submatvec, (inp, mat, vec.t().contiguous().t()), {}, (B, n)),
        ("sym_solve streamed", nfm.sym_solve, (mat, vec), {}, (B, n)),
        ("sym_solve per-voxel", nfm.sym_solve, (mat, vec, vec.abs()), {"method": "lu"}, (B, n)),
        ("sym_solve scalar", nfm.sym_solve, (mat, vec, 0.5), {}, (B, n)),
        ("sym_solve broadcast", nfm.sym_solve, (mat[:1], vec), {}, (B, n)),
        ("sym_invert streamed", nfm.sym_invert, (mat,), {}, (B, nn)),
        ("sym_invert diag streamed", nfm.sym_invert, (mat, True), {}, (B, n)),
        ("sym_invert half", nfm.sym_invert, (half,), {}, (B, nn)),
        ("batchinv streamed", nfm.batchinv, (a,), {}, (B, n, n)),
        ("batchinv strided", nfm.batchinv, (a[::2],), {}, (len(range(0, B, 2)), n, n)),
        ("batchdet streamed", nfm.batchdet, (a,), {}, (B,)),
        ("batchdet strided", nfm.batchdet, (a.transpose(-1, -2),), {}, (B,)),
        ("batchmatvec", nfm.batchmatvec, (a, vec), {}, (B, n)),
        ("lmdiv streamed", nfm.lmdiv, (a, rhs), {}, (B, n, 3)),
        ("lmdiv broadcast", nfm.lmdiv, (a[:1], rhs), {}, (B, n, 3)),
        ("rmdiv", nfm.rmdiv, (rhs.transpose(-1, -2), a), {}, (B, 3, n)),
        ("inv streamed", nfm.inv, (a,), {}, (B, n, n)),
        ("solvevec streamed", nfm.solvevec, (a, vec), {}, (B, n)),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("n,dtype", [(3, torch.float32), (6, torch.float64)], ids=["n3_f32", "n6_f64"])
def test_wrong_shape_out_is_rejected_on_every_route(n, dtype):
    """Fewer / more rows, a wider / narrower record, an extra leading dim: RuntimeError with the
    device path's message, out untouched, nothing launched, inputs unchanged."""
    for name, fn, args, kw, shape in _out_routes(n, dtype):
        _rejects(fn, args, kw, shape, dtype)
        got = fn(*args, **kw)                       # and the right shape is the result's
        assert tuple(got.shape) == shape, name


# --------------------------------------------------------------------------
# batches of a million or more at the default chunk size
# --------------------------------------------------------------------------

@pytest.mark.gpu
def test_million_matrix_batches_at_the_default_chunk():
    """Many default-size chunks: every matrix checked in float64 on the GPU, bits against the device call."""
    nfm = _nfm()
    b = 1_048_583
    mat = G.spd_packed(b, 3, torch.float64, 1).pin_memory()
    vec, reg = G.vectors(b, 3, torch.float64, 2).pin_memory(), (G.vectors(b, 3, torch.float64, 3).abs() + 0.1).pin_memory()
    x = nfm.sym_solve(mat, vec, reg)
    dm, dv, dr = mat.to(DEV), vec.to(DEV), reg.to(DEV)
    assert torch.equal(x, nfm.sym_solve(dm, dv, dr).cpu())
    assert worst_err(x.to(DEV), _solve(_full(dm, 3) + torch.diag_embed(dr), dv)) <= TOL[torch.float64]
    del mat, vec, reg, dm, dv, dr, x
    b = 1_000_003
    a = G.dense_shifted(b, 4, torch.float64, 4).pin_memory()
    inv = nfm.batchinv(a)
    da = a.to(DEV)
    assert torch.equal(inv, nfm.batchinv(da).cpu())
    assert worst_err(inv.to(DEV), torch.linalg.inv(da), 2) <= TOL[torch.float64]
    del inv
    a = G.dense_shifted(b, 3, torch.float32, 5).pin_memory()
    rhs = G.vectors((b, 3), 5, torch.float32, 6).pin_memory()
    x = nfm.lmdiv(a, rhs)
    da, dr = a.to(DEV), rhs.to(DEV)
    assert torch.equal(x, nfm.lmdiv(da, dr).cpu())
    assert worst_err(x.to(DEV), torch.linalg.solve(da.double(), dr.double()), 2) <= TOL[torch.float32]


# --------------------------------------------------------------------------
# NFM_HOST_CHUNK_MB / NFM_HOST_NBUF, read at import: child processes
# --------------------------------------------------------------------------

SETTINGS_B = 400_009


def _settings_jobs():
    """name -> (call, dtype, input record elems, output record elems) on seeded pinned CPU inputs."""
    nfm = _nfm()
    B = SETTINGS_B
    m3, v3 = G.spd_packed(B, 3, torch.float32, 1).pin_memory(), G.vectors(B, 3, torch.float32, 2).pin_memory()
    i3 = G.vectors(B, 3, torch.float32, 3).pin_memory()
    m6 = G.spd_packed(B, 6, torch.float64, 4).pin_memory()
    a4 = G.dense_shifted(B, 4, torch.float64, 5).pin_memory()
    r4 = G.vectors((B, 4), 5, torch.float64, 6).pin_memory()
    a10 = G.dense_shifted(B, 10, torch.float32, 7).pin_memory()
    return {
        "solve3_f32": (lambda: nfm.sym_solve(m3, v3, i3.abs()), torch.float32, 12, 3),
        "submatvec3_f32": (lambda: nfm.sym_submatvec(i3, m3, v3), torch.float32, 12, 3),
        "invert6_diag_f64": (lambda: nfm.sym_invert(m6, True, method="lu"), torch.float64, 21, 6),
        "batchinv4_f64": (lambda: nfm.batchinv(a4), torch.float64, 16, 16),
        "lmdiv4x5_f64": (lambda: nfm.lmdiv(a4, r4), torch.float64, 36, 20),
        "batchdet10_f32": (lambda: nfm.batchdet(a10), torch.float32, 100, 1),
    }


def _digest(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def run_settings_jobs():
    from nitorch_fastmath_b200 import _host
    res = {}
    for name, (call, dtype, ie, oe) in _settings_jobs().items():
        before = _lib.launch_count()
        out = call()
        res[name] = dict(digest=_digest(out), launches=_lib.launch_count() - before,
                         chunks=-(-SETTINGS_B // _host.chunk_for(dtype, ie, oe)))
    return res


def _child_main(argv):
    from nitorch_fastmath_b200 import _host
    res = run_settings_jobs()
    res["_settings"] = dict(chunk_bytes=_host._DEFAULT_CHUNK_BYTES, nbuf=_host._NBUF)
    with open(argv[0], "w") as f:
        json.dump(res, f)


@pytest.fixture(scope="module")
def default_settings_digests():
    return run_settings_jobs()


@pytest.mark.gpu
@pytest.mark.parametrize("nbuf", [1, 2, 5])
def test_pipeline_settings_in_a_child_process(tmp_path, default_settings_digests, nbuf):
    """1 MB chunks on 1, 2 or 5 buffers: many chunks, the ring wraps at least twice, and every
    result has the bits of the default 16 MB / 3 buffers."""
    dest = str(tmp_path / "child.json")
    env = dict(os.environ, NFM_HOST_CHUNK_MB="1", NFM_HOST_NBUF=str(nbuf))
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    code = "import sys, test_host_path as T; T._child_main(sys.argv[1:])"
    r = subprocess.run([sys.executable, "-c", code, dest], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    with open(dest) as f:
        child = json.load(f)
    assert child.pop("_settings") == dict(chunk_bytes=1 << 20, nbuf=nbuf)
    assert set(child) == set(default_settings_digests)
    for name, c in child.items():
        assert c["chunks"] >= 2 * nbuf + 1 and c["chunks"] > default_settings_digests[name]["chunks"], (name, c)
        assert c["launches"] >= c["chunks"], (name, c)
        assert c["digest"] == default_settings_digests[name]["digest"], (name, nbuf)


# --------------------------------------------------------------------------
# concurrency and state
# --------------------------------------------------------------------------

@pytest.mark.gpu
def test_two_threads_share_the_device_pipeline():
    """Two threads run host calls of different record sizes on one device at once: the shared
    workspace grows between calls under the device lock, and both results stay exact."""
    from nitorch_fastmath_b200 import _host
    nfm = _nfm()
    st = _host._state(torch.device(DEV))
    with st.lock:
        st.workspace = None
    m3, v3 = G.spd_packed(300_007, 3, torch.float32, 1).pin_memory(), G.vectors(300_007, 3, torch.float32, 2).pin_memory()
    m10 = G.spd_packed(200_003, 10, torch.float64, 3).pin_memory()
    want3 = nfm.sym_solve(m3.to(DEV), v3.to(DEV)).cpu()
    want10 = nfm.sym_invert(m10.to(DEV)).cpu()
    errors = []

    def loop(fn, want):
        try:
            torch.cuda.set_device(0)
            for _ in range(4):
                got = fn()
                if not torch.equal(got, want):
                    errors.append("mismatch")
        except Exception as e:          # noqa: BLE001 - reported in the main thread
            errors.append(repr(e))

    threads = [threading.Thread(target=loop, args=(lambda: nfm.sym_solve(m3, v3), want3)),
               threading.Thread(target=loop, args=(lambda: nfm.sym_invert(m10), want10))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert errors == []
    assert st.workspace.numel() >= _lib.load().nfm_host_workspace_bytes(
        _lib.F64, _host.chunk_for(torch.float64, 55, 55), _host._NBUF, 55, 55)


@pytest.mark.gpu
def test_workspace_grows_and_is_reused():
    """A small call, a large one (the workspace reallocates), a small one again: all exact."""
    from nitorch_fastmath_b200 import _host
    nfm = _nfm()
    st = _host._state(torch.device(DEV))
    with st.lock:
        st.workspace = None
    small = G.spd_packed(5000, 3, torch.float32, 1).pin_memory()
    big = G.spd_packed(400_000, 10, torch.float64, 2).pin_memory()
    want_s = nfm.sym_invert(small.to(DEV)).cpu()
    assert torch.equal(nfm.sym_invert(small), want_s)
    size_small = st.workspace.numel()
    assert torch.equal(nfm.sym_invert(big), nfm.sym_invert(big.to(DEV)).cpu())
    assert st.workspace.numel() > size_small
    assert torch.equal(nfm.sym_invert(small), want_s)


@pytest.mark.gpu
def test_host_call_after_queued_device_work():
    """The pipeline streams wait for the current stream: a pinned CPU operand that a queued
    non-blocking device-to-host copy is still filling is read only after the copy lands."""
    nfm = _nfm()
    b, n = 200_003, 6
    dm = G.spd_packed(b, n, torch.float32, 1).to(DEV)
    dv = G.vectors(b, n, torch.float32, 2).to(DEV)
    want = nfm.sym_solve(dm, dv).cpu()
    hm = torch.full((b, _pk(n)), float("nan")).pin_memory()
    hv = torch.full((b, n), float("nan")).pin_memory()
    torch.cuda.synchronize()
    torch.cuda._sleep(50_000_000)                    # keep the current stream busy for a few ms
    hm.copy_(dm, non_blocking=True)
    hv.copy_(dv, non_blocking=True)
    got = nfm.sym_solve(hm, hv)
    assert torch.equal(got, want)


# --------------------------------------------------------------------------
# multi_gpu: one slab per device, each through its own pipeline
# --------------------------------------------------------------------------

def _multi_devices():
    return [[0]] + ([list(range(torch.cuda.device_count()))] if torch.cuda.device_count() > 1 else [None])


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["device0", "all"])
def test_multi_gpu_functions(which):
    devices = _multi_devices()[0 if which == "device0" else 1]
    if devices is None:
        pytest.skip("one visible GPU")
    from nitorch_fastmath_b200 import multi_gpu
    nfm = _nfm()
    b = 1_000_003                                   # slab bounds are not multiples of any chunk
    mat = G.spd_packed(b, 4, torch.float32, 1).pin_memory()
    vec, reg = G.vectors(b, 4, torch.float32, 2).pin_memory(), (G.vectors(b, 4, torch.float32, 3).abs() + 0.1).pin_memory()
    dm, dv, dr = mat.to(DEV), vec.to(DEV), reg.to(DEV)
    for method in (None, "lu"):
        assert torch.equal(multi_gpu.sym_solve_multi(mat, vec, reg, devices=devices, method=method),
                           nfm.sym_solve(dm, dv, dr, method=method).cpu())
    out = torch.empty_like(vec).pin_memory()
    r = multi_gpu.sym_solve_multi(mat, vec, devices=devices, out=out)
    assert r.data_ptr() == out.data_ptr() and torch.equal(out, nfm.sym_solve(dm, dv).cpu())
    for diag in (False, True):
        want = nfm.sym_invert(dm, diag, method="lu").cpu()
        assert torch.equal(multi_gpu.sym_invert_multi(mat, diag, devices=devices, method="lu"), want)
        out = torch.empty(want.shape).pin_memory()
        assert multi_gpu.sym_invert_multi(mat, diag, devices=devices, out=out, method="lu") is out
        assert torch.equal(out, want)
    out = torch.empty_like(vec)
    assert multi_gpu.sym_matvec_multi(mat, vec, devices=devices, out=out) is out
    assert torch.equal(out, nfm.sym_matvec(dm, dv).cpu())
    assert worst_err(out, (_full(mat, 4) @ vec.double()[..., None])[..., 0]) <= TOL[torch.float32]


@pytest.mark.gpu
def test_multi_gpu_rejects_a_wrong_out_before_any_slab():
    from nitorch_fastmath_b200 import multi_gpu
    b, n = 10_007, 3
    mat = G.spd_packed(b, n, torch.float32, 1).pin_memory()
    vec = G.vectors(b, n, torch.float32, 2).pin_memory()
    for fn, args, kw, shape in ((multi_gpu.sym_solve_multi, (mat, vec), {}, (b, n)),
                                (multi_gpu.sym_matvec_multi, (mat, vec), {}, (b, n)),
                                (multi_gpu.sym_invert_multi, (mat,), {}, (b, _pk(n))),
                                (multi_gpu.sym_invert_multi, (mat, True), {}, (b, n))):
        _rejects(fn, args, dict(kw, devices=[0]), shape, torch.float32)
    with pytest.raises(ValueError):
        multi_gpu.sym_solve_multi(mat, vec, devices=[0], out=torch.empty(b, n, device=DEV))


# --------------------------------------------------------------------------
# bench.py's end-to-end call
# --------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["sym_solve3", "sym_solve6", "sym_invert6", "sym_solve10", "sym_matvec3",
                                      "dense_inv4_f64", "dense_det4_f64", "dense_solve4_f64"])
def test_bench_end_to_end_call_is_the_device_result(workload):
    """bench.api_call on pinned CPU inputs and an out shaped as bench.py shapes it: the bits of
    the same call on the device."""
    import bench
    w = bench.WORKLOADS[workload]
    kind, n = w["kind"], w["n"]
    dtype = torch.float32 if w["dtype"] == "f32" else torch.float64
    slab = 200_003
    ins = bench.make_inputs(kind, n, dtype, slab, DEV, seed=bench.operand_seed(0, 0))
    _, olen = bench.record_lengths(kind, n)
    host_in = [t.cpu().pin_memory() for t in ins]

    def shaped(device):
        o = torch.empty((slab, olen) if olen > 1 else (slab,), dtype=dtype, device=device)
        return o.view(slab, n, n) if kind == "batch_inv" else o
    host_out = shaped("cpu").pin_memory()
    dev_out = shaped(DEV)
    r = bench.api_call(kind, host_in, host_out)
    assert r.data_ptr() == host_out.data_ptr() and r.device.type == "cpu"
    bench.api_call(kind, ins, dev_out)
    assert torch.equal(host_out, dev_out.cpu())
