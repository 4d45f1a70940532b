"""Every bulk kernel in the state it runs in on full-size volumes.

The parity tests run batches of a few thousand matrices: the TMA tile kernel, the
warp-pool kernel and the many-right-hand-sides kernel never reuse a stage, buffer or
ring slot there, and light ops never reach their large-batch tile geometry
(``Tune`` above ``TuneSmall::kBelowBytes``).  Here every case is sized from the launch
record of the library (``nfm_last_launch_shape``), not from copied constants:

* small geometry: a batch below the switch on which every CTA passes its ring of
  stages at least twice (tile kernel: tiles >= (2 stages + 1) x grid; pool kernel:
  warp tiles >= 3 x buffers x grid; many right-hand sides: warp tiles >= 3 x depth x
  warps x grid), with a partial last tile and a few matrices past the 16-byte granule;
* large geometry (light ops that have two): the batch doubled until the geometry
  switches, then grown until the ring wraps twice there as well.

Inputs are distinct per matrix (a record read from the wrong stage is an O(1) error),
every matrix is checked against a float64 reference on the GPU, slices at the start,
middle and end against the CPU oracle, and the large-geometry result must equal, bit
for bit, the same call cut into chunks that run in the small geometry.

The path switches of README (NFM_BALANCE, NFM_DISABLE_PDL, ...) are read once per
process, so they are exercised in a child process.
"""
from __future__ import annotations

import hashlib
import json
import os
import subprocess
import sys
import threading
from dataclasses import dataclass, field
from typing import Callable, Optional

import numpy as np
import pytest
import torch

from conftest import ROOT, TOL
from oracle import ref_port as P

DEV = "cuda:0"
CHUNK = 2 << 20                    # float64 reference / input generation in chunks of this many matrices
SLICE = 20_000                     # CPU-oracle slices
STOP_BYTES = 640 << 20             # operand bytes past which no light op keeps its small geometry
DTYPES = [torch.float32, torch.float64]
COVERAGE: list = []                # rows of the coverage table (printed at the end of the module)


# --------------------------------------------------------------------------
# launch record (runs without a GPU)
# --------------------------------------------------------------------------

def test_launch_shape_hook_exists_and_starts_empty():
    """nfm_last_launch_shape is exported, bound, thread-local, and reports kind 0
    on a thread that has launched nothing; a NULL output is rejected."""
    from nitorch_fastmath_b200 import _lib
    lib = _lib.load()
    assert "nfm_last_launch_shape" in _lib.SIGNATURES
    got = {}
    t = threading.Thread(target=lambda: got.update(_lib.last_launch_shape()))
    t.start()
    t.join()
    assert got == dict.fromkeys(_lib.LAUNCH_FIELDS, 0)
    assert lib.nfm_last_launch_shape(None) == -2


# --------------------------------------------------------------------------
# inputs: generated on the GPU in chunks, distinct per matrix
# --------------------------------------------------------------------------

def _tri(n):
    return torch.triu_indices(n, n, 1, device=DEV)


def _pack(full):
    n = full.shape[-1]
    iu = _tri(n)
    return torch.cat([full.diagonal(0, -1, -2), full[..., iu[0], iu[1]]], -1)


def _unpack(mat, n):
    idx = torch.empty(n, n, dtype=torch.long)
    for i in range(n):
        for j in range(n):
            idx[i, j] = P.packed_index(n, i, j)
    return mat[..., idx.to(mat.device)]


def _chunked(batch, dtype, shape, fill, seed):
    out = torch.empty(batch, *shape, device=DEV, dtype=dtype)
    g = torch.Generator(device=DEV).manual_seed(seed)
    for c in range(0, batch, CHUNK):
        m = min(CHUNK, batch - c)
        out[c:c + m] = fill(m, g).to(dtype)
    return out


def spd(batch, n, dtype, seed):
    def fill(m, g):
        a = torch.randn(m, n, n, device=DEV, dtype=torch.float64, generator=g)
        full = a @ a.transpose(-1, -2)
        full.diagonal(0, -1, -2).add_(n)
        return _pack(full)
    return _chunked(batch, dtype, (n * (n + 1) // 2,), fill, seed)


def spd_or_indefinite(batch, n, dtype, seed):
    """Every second matrix symmetric indefinite, H diag(+-[1, 2]) H (H a Householder
    reflection): the checked LDL^T falls back to pivoted LU in some lanes only."""
    def fill(m, g):
        a = torch.randn(m, n, n, device=DEV, dtype=torch.float64, generator=g)
        full = a @ a.transpose(-1, -2)
        full.diagonal(0, -1, -2).add_(n)
        v = torch.randn(m, n, 1, device=DEV, dtype=torch.float64, generator=g)
        h = torch.eye(n, device=DEV, dtype=torch.float64) - 2 * (v @ v.transpose(-1, -2)) / (v * v).sum((-1, -2), keepdim=True)
        lam = 1 + torch.rand(m, n, device=DEV, dtype=torch.float64, generator=g)
        lam = lam * torch.where(torch.arange(n, device=DEV) % 2 == 0, 1.0, -1.0)
        ind = (h * lam[..., None, :]) @ h
        full[1::2] = ind[1::2]
        return _pack(full)
    return _chunked(batch, dtype, (n * (n + 1) // 2,), fill, seed)


def vecs(batch, n, dtype, seed, k=None, positive=False):
    shape = (n,) if k is None else (n, k)

    def fill(m, g):
        x = torch.randn(m, *shape, device=DEV, dtype=torch.float64, generator=g)
        return x.abs() + 0.1 if positive else x
    return _chunked(batch, dtype, shape, fill, seed)


def dense(batch, n, dtype, seed):
    """randn + 10 I; every second matrix with its rows shuffled, so partial pivoting
    exchanges rows in some lanes of a warp and not in others."""
    def fill(m, g):
        a = torch.randn(m, n, n, device=DEV, dtype=torch.float64, generator=g)
        a.diagonal(0, -1, -2).add_(10)
        if n > 1:
            perm = torch.rand(m, n, device=DEV, generator=g).argsort(-1)
            shuffled = a.gather(-2, perm[..., None].expand(m, n, n))
            a[1::2] = shuffled[1::2]
        return a
    return _chunked(batch, dtype, (n, n), fill, seed)


def dense_spd(batch, n, dtype, seed):
    def fill(m, g):
        a = torch.randn(m, n, n, device=DEV, dtype=torch.float64, generator=g)
        full = a @ a.transpose(-1, -2)
        full.diagonal(0, -1, -2).add_(n)
        return full
    return _chunked(batch, dtype, (n, n), fill, seed)


# --------------------------------------------------------------------------
# float64 references (the formulas of include/nfm.h)
# --------------------------------------------------------------------------

def _full(mat, n, layout):
    mat = mat.double()
    if layout == "S":
        return _unpack(mat, n)
    if layout == "D":
        return torch.diag_embed(mat)
    return torch.diag_embed(mat.expand(*mat.shape[:-1], n))


def _solve(a, b):
    return torch.linalg.solve(a, b[..., None])[..., 0]


def _outer2(u, w, layout):
    u, w = u.double(), w.double()
    if layout == "E":
        return (u * w).sum(-1, keepdim=True)
    if layout == "D":
        return u * w
    s = u[..., :, None] * w[..., None, :]
    return _pack(s + s.transpose(-1, -2) - torch.diag_embed(u * w))


def _invert_backward(inv, grad, n, diag_only):
    b = _unpack(inv.double(), n)
    if diag_only:
        g = torch.diag_embed(grad.double())
    else:
        g = _unpack(grad.double(), n)
        g = (g + torch.diag_embed(g.diagonal(0, -1, -2))) / 2
    m = b @ g @ b
    return -(2 * _pack(m) - torch.cat([m.diagonal(0, -1, -2), torch.zeros_like(_pack(m)[..., n:])], -1))


def _det_backward(mat, grad, n):
    a = _unpack(mat.double(), n)
    adj = torch.linalg.det(a)[..., None, None] * torch.linalg.inv(a)
    out = 2 * _pack(adj)
    out[..., :n] = adj.diagonal(0, -1, -2)
    return out * grad.double()[..., None]


def _ghat(g, n):
    """The full symmetric form of a packed gradient with the off-diagonals halved."""
    f = _unpack(g.double(), n)
    return (f + torch.diag_embed(f.diagonal(0, -1, -2))) / 2


def _pack2(m):
    """M_ii, 2 M_ij (i < j) of a symmetric M."""
    return _pack(2 * m - torch.diag_embed(m.diagonal(0, -1, -2)))


def _matmul_backward(i, k, d, which):
    """dJ (flattened) and / or dH of J^T H J (J H J^T for k = d <= 3), one record [dJ | dH]."""
    j = i["j"].double()
    mode1 = k == d and k <= 3
    h, gh = _unpack(i["h"].double(), d if mode1 else k), _ghat(i["g"], k if mode1 else d)
    parts = []
    if which & 1:
        parts.append((2 * gh @ j @ h if mode1 else 2 * h @ j @ gh).flatten(-2))
    if which & 2:
        parts.append(_pack2(j.transpose(-1, -2) @ gh @ j if mode1 else j @ gh @ j.transpose(-1, -2)))
    return torch.cat(parts, -1)


# --------------------------------------------------------------------------
# the case table
# --------------------------------------------------------------------------

@dataclass
class Case:
    name: str
    dtype: torch.dtype
    gen: Callable            # (batch, seed) -> dict of per-matrix device tensors
    run: Callable            # (ins) -> output
    ref: Callable            # (ins) -> float64 output
    rec: int = 1             # record dims of the output (per-matrix norm-wise error)
    scale: float = 1.0
    addend: Optional[str] = None          # inp +/- A v: error relative to |addend| + |A v|
    oracle: Optional[Callable] = None     # (cpu ins) -> output of oracle/ref_port.py
    oracle_rows: int = SLICE
    extra: dict = field(default_factory=dict)

    def __str__(self):
        return self.name


def _nfm():
    import nitorch_fastmath_b200 as pkg
    return pkg


def _sym_cases():
    nfm = _nfm()
    from nitorch_fastmath_b200 import _autograd as A
    from nitorch_fastmath_b200 import _lib
    lay_code = {"S": _lib.LAYOUT_SYM, "D": _lib.LAYOUT_DIAG, "E": _lib.LAYOUT_SCALED_IDENTITY}
    cases = []
    for dt in DTYPES:
        t = "f32" if dt == torch.float32 else "f64"
        for n in range(1, 11):
            nn = n * (n + 1) // 2
            mlen = {"S": nn, "D": n, "E": 1}
            for lay in "SDE":
                if lay != "S" and n == 1:
                    continue
                L = mlen[lay]

                def mk_mat(b, s, L=L, n=n, lay=lay, dt=dt):
                    return spd(b, n, dt, s) if lay == "S" else vecs(b, L, dt, s, positive=True)

                if lay == "S":
                    cases.append(Case(f"matvec_{lay}_{t}_n{n}", dt,
                                  lambda b, s, n=n, dt=dt, mk=mk_mat: dict(mat=mk(b, s), vec=vecs(b, n, dt, s + 1)),
                                  lambda i: nfm.sym_matvec(i["mat"], i["vec"]),
                                  lambda i, n=n, lay=lay: (_full(i["mat"], n, lay) @ i["vec"].double()[..., None])[..., 0],
                                  oracle=lambda i: P.sym_matvec(i["mat"], i["vec"])))
                # (sym_submatvec is the same instantiation with the sign flag)
                cases.append(Case(f"addmatvec_{lay}_{t}_n{n}", dt,
                                  lambda b, s, n=n, dt=dt, mk=mk_mat: dict(inp=vecs(b, n, dt, s + 2), mat=mk(b, s), vec=vecs(b, n, dt, s + 1)),
                                  lambda i: nfm.sym_addmatvec(i["inp"], i["mat"], i["vec"]),
                                  lambda i, n=n, lay=lay: i["inp"].double() + (_full(i["mat"], n, lay) @ i["vec"].double()[..., None])[..., 0],
                                  addend="inp"))
                regs = [("voxel", "field")]
                if lay == "S":
                    regs += [("none", None), ("bcast", [0.5, 0.25, 0.125][: min(n, 3)] if n <= 3 else 0.25)]
                methods = [None] if lay != "S" or n <= 4 else [None, "ldl", "lu", "warp"]
                for method in methods:
                    for rname, reg in regs:
                        if (method == "ldl" and rname != "voxel") or (method in ("lu", "warp") and rname != "none"):
                            continue
                        # (indefinite only without a per-voxel shift, which could move an eigenvalue onto 0)
                        ind = lay == "S" and method in (None, "lu") and rname != "voxel"

                        def g_solve(b, s, n=n, dt=dt, mk=mk_mat, reg=reg, ind=ind):
                            d = dict(mat=spd_or_indefinite(b, n, dt, s) if ind else mk(b, s), vec=vecs(b, n, dt, s + 1))
                            if reg == "field":
                                d["reg"] = vecs(b, n, dt, s + 3, positive=True)
                            return d

                        def r_solve(i, n=n, lay=lay, reg=reg):
                            a = _full(i["mat"], n, lay)
                            if reg == "field":
                                a = a + torch.diag_embed(i["reg"].double())
                            elif reg is not None:
                                a = a + torch.diag_embed(torch.as_tensor(reg, dtype=torch.float64, device=DEV).expand(n))
                            return _solve(a, i["vec"].double())

                        def run_solve(i, reg=reg, method=method):
                            d = i["reg"] if reg == "field" else reg
                            return nfm.sym_solve(i["mat"], i["vec"], d, method=method)

                        def o_solve(i, reg=reg, method=method):
                            d = i["reg"] if reg == "field" else reg
                            return P.sym_solve(i["mat"], i["vec"], d)

                        cases.append(Case(f"solve_{lay}_{method or 'auto'}_{rname}_{t}_n{n}", dt, g_solve, run_solve, r_solve,
                                          scale=20 if ind else 1, oracle=o_solve if lay == "S" and method is None else None,
                                          extra=dict(warp=method == "warp" and n >= 5)))
            # sym_invert: full and diag=True; auto / ldl / lu
            for method in ([None] if n <= 4 else [None, "ldl", "lu"]):
                for diag in ((False, True) if method is None else (False,)):
                    ind = method in (None, "lu") and n > 4
                    gi = (lambda b, s, n=n, dt=dt, ind=ind: dict(mat=spd_or_indefinite(b, n, dt, s) if ind else spd(b, n, dt, s)))

                    def r_inv(i, n=n, diag=diag):
                        inv = torch.linalg.inv(_unpack(i["mat"].double(), n))
                        return inv.diagonal(0, -1, -2) if diag else _pack(inv)

                    cases.append(Case(f"invert_{'diag_' if diag else ''}{method or 'auto'}_{t}_n{n}", dt, gi,
                                      lambda i, diag=diag, method=method: nfm.sym_invert(i["mat"], diag, method=method), r_inv,
                                      scale=20 if ind else 1,
                                      oracle=(lambda i, diag=diag: P.sym_invert(i["mat"], diag)) if method is None else None,
                                      oracle_rows=SLICE if n <= 6 else 4000))
            gm = (lambda b, s, n=n, dt=dt: dict(mat=spd(b, n, dt, s)))
            cases.append(Case(f"det_{t}_n{n}", dt, gm, lambda i: nfm.sym_det(i["mat"]),
                              lambda i, n=n: torch.linalg.det(_unpack(i["mat"].double(), n)), rec=0, scale=10,
                              oracle=lambda i: P.sym_det(i["mat"])))
            cases.append(Case(f"to_full_{t}_n{n}", dt, gm, lambda i: nfm.sym_to_full(i["mat"]),
                              lambda i, n=n: _unpack(i["mat"].double(), n), rec=2, oracle=lambda i: P.sym_to_full(i["mat"])))
            cases.append(Case(f"outer_{t}_n{n}", dt, lambda b, s, n=n, dt=dt: dict(vec=vecs(b, n, dt, s)),
                              lambda i: nfm.sym_outer(i["vec"]),
                              lambda i: _pack(i["vec"].double()[..., :, None] * i["vec"].double()[..., None, :]),
                              oracle=lambda i: P.sym_outer(i["vec"])))
            for diag in (False, True):
                def g_upd(b, s, n=n, dt=dt, diag=diag):
                    d = dict(x=vecs(b, n, dt, s + 2), mat=spd(b, n, dt, s), vec=vecs(b, n, dt, s + 1))
                    if diag:
                        d["reg"] = vecs(b, n, dt, s + 3, positive=True)
                    return d

                def r_upd(i, n=n, diag=diag):
                    a = _unpack(i["mat"].double(), n) + 0.3 * torch.eye(n, device=DEV, dtype=torch.float64)
                    if diag:
                        a = a + torch.diag_embed(i["reg"].double())
                    return i["x"].double() - 0.5 * _solve(a, i["vec"].double())

                cases.append(Case(f"solve_update_{'diag_' if diag else ''}{t}_n{n}", dt, g_upd,
                                  lambda i: nfm.sym_solve_update(i["x"], i["mat"], i["vec"], 0.3, 0.5, diag=i.get("reg")),
                                  r_upd, addend="x"))
            # backward kernels
            for lay in "SDE":
                cases.append(Case(f"outer2_{lay}_{t}_n{n}", dt,
                                  lambda b, s, n=n, dt=dt: dict(u=vecs(b, n, dt, s), w=vecs(b, n, dt, s + 1)),
                                  lambda i, lay=lay: A.outer2(i["u"], i["w"], lay_code[lay], -1),
                                  lambda i, lay=lay: -_outer2(i["u"], i["w"], lay),
                                  extra=dict(dot=lay == "E")))
            for diag in (False, True):
                cases.append(Case(f"invert_backward_{'diag_' if diag else ''}{t}_n{n}", dt,
                                  lambda b, s, n=n, nn=nn, dt=dt, diag=diag: dict(inv=spd(b, n, dt, s), g=vecs(b, n if diag else nn, dt, s + 1)),
                                  lambda i, diag=diag: A.invert_backward(i["inv"], i["g"], diag),
                                  lambda i, n=n, diag=diag: _invert_backward(i["inv"], i["g"], n, diag), scale=10))
            cases.append(Case(f"det_backward_{t}_n{n}", dt,
                              lambda b, s, n=n, dt=dt: dict(mat=spd(b, n, dt, s), g=vecs(b, 1, dt, s + 1)[:, 0].contiguous()),
                              lambda i: A.det_backward(i["mat"], i["g"]),
                              lambda i, n=n: _det_backward(i["mat"], i["g"], n), scale=10 * n))
        # the fused Gauss-Newton builders at their register-kernel shapes
        for k, d in ((1, 1), (2, 2), (3, 3), (4, 4), (6, 6), (3, 2), (2, 3), (10, 3)):
            def g_mm(b, s, k=k, d=d, dt=dt):
                j = vecs(b, k, dt, s, k=d)
                j = 0.3 * j + 2 * torch.eye(k, d, device=DEV, dtype=dt)
                return dict(j=j, h=spd(b, k, dt, s + 1), g=vecs(b, d, dt, s + 2), reg=vecs(b, d, dt, s + 3, positive=True) + (1.0 if k < d else 0.0))

            def r_mm(i, k=k, d=d):
                j, h = i["j"].double(), _unpack(i["h"].double(), k)
                return j @ h @ j.transpose(-1, -2) if (k == d and k <= 3) else j.transpose(-1, -2) @ h @ j

            cases.append(Case(f"matmul_{t}_k{k}_d{d}", dt, g_mm, lambda i: nfm.sym_matmul(i["j"], i["h"]),
                              lambda i, r=r_mm: _pack(r(i)), scale=4))
            cases.append(Case(f"matmul_solve_{t}_k{k}_d{d}", dt, g_mm, lambda i: nfm.sym_matmul_solve(i["j"], i["h"], i["g"], i["reg"]),
                              lambda i, r=r_mm: _solve(r(i) + torch.diag_embed(i["reg"].double()), i["g"].double()), scale=10))
    return cases


def _dense_cases():
    nfm = _nfm()
    cases = []
    for dt in DTYPES:
        t = "f32" if dt == torch.float32 else "f64"
        for n in range(1, 11):
            ga = (lambda b, s, n=n, dt=dt: dict(a=dense(b, n, dt, s)))
            gs = (lambda b, s, n=n, dt=dt: dict(a=dense_spd(b, n, dt, s)))
            inv = lambda i: torch.linalg.inv(i["a"].double())
            cases.append(Case(f"batchinv_{t}_n{n}", dt, ga, lambda i: nfm.batchinv(i["a"]), inv, rec=2, scale=4,
                              oracle=lambda i: P.batchinv(i["a"]), oracle_rows=SLICE if n <= 6 else 4000))
            if n <= 3:   # (from order 4 on the same kernel as batchinv)
                cases.append(Case(f"inv_lu_{t}_n{n}", dt, ga, lambda i: nfm.inv(i["a"], "lu"), inv, rec=2, scale=4))
            cases.append(Case(f"inv_chol_{t}_n{n}", dt, gs, lambda i: nfm.inv(i["a"], "chol"), inv, rec=2, scale=4))
            cases.append(Case(f"batchdet_{t}_n{n}", dt, ga, lambda i: nfm.batchdet(i["a"]),
                              lambda i: torch.linalg.det(i["a"].double()), rec=0, scale=4, oracle=lambda i: P.batchdet(i["a"])))
            gav = (lambda b, s, n=n, dt=dt: dict(a=dense(b, n, dt, s), b=vecs(b, n, dt, s + 1)))
            cases.append(Case(f"batchmatvec_{t}_n{n}", dt, gav, lambda i: nfm.batchmatvec(i["a"], i["b"]),
                              lambda i: (i["a"].double() @ i["b"].double()[..., None])[..., 0]))
            cases.append(Case(f"solvevec_{t}_n{n}", dt, gav, lambda i: nfm.solvevec(i["a"], i["b"]),
                              lambda i: _solve(i["a"].double(), i["b"].double()), scale=4,
                              oracle=lambda i: P.solvevec(i["a"], i["b"])))
            for k in (2, 4, 5, 12):
                for meth in (("lu", "chol") if k == 5 else ("lu",)):
                    g_lm = (lambda b, s, n=n, dt=dt, k=k, meth=meth:
                            dict(a=dense_spd(b, n, dt, s) if meth == "chol" else dense(b, n, dt, s), b=vecs(b, n, dt, s + 1, k=k)))
                    cases.append(Case(f"lmdiv_{meth}_k{k}_{t}_n{n}", dt, g_lm, lambda i, meth=meth: nfm.lmdiv(i["a"], i["b"], meth),
                                      lambda i: torch.linalg.solve(i["a"].double(), i["b"].double()), rec=2, scale=4,
                                      extra=dict(many=k > 4)))
            for k in (1, 9):
                g_rm = (lambda b, s, n=n, dt=dt, k=k: dict(a=dense(b, n, dt, s), r=vecs(b, k, dt, s + 1, k=n)))
                cases.append(Case(f"rmdiv_k{k}_{t}_n{n}", dt, g_rm, lambda i: nfm.rmdiv(i["r"], i["a"]),
                                  lambda i: i["r"].double() @ torch.linalg.inv(i["a"].double()), rec=2, scale=4,
                                  extra=dict(many=True)))
    return cases


MATMUL_SHAPES = ((1, 1), (2, 2), (3, 3), (4, 4), (6, 6), (3, 2), (2, 3), (10, 3))


def _grad_cases():
    """The backward kernels of the dense routines and of the Gauss-Newton builders (_autograd.py)."""
    from nitorch_fastmath_b200 import _autograd as A
    from nitorch_fastmath_b200 import _lib
    cases = []
    for dt in DTYPES:
        t = "f32" if dt == torch.float32 else "f64"
        es = torch.finfo(dt).bits // 8
        for n in range(1, 11):
            nn = n * (n + 1) // 2
            for sym in (False, True):
                def g_inv(b, s, n=n, dt=dt, sym=sym):
                    return dict(y=dense_spd(b, n, dt, s) if sym else dense(b, n, dt, s), g=vecs(b, n, dt, s + 1, k=n))

                def r_inv(i, sym=sym):
                    y, g = i["y"].double(), i["g"].double()
                    if sym:
                        return -y @ ((g + g.transpose(-1, -2)) / 2) @ y
                    return -y.transpose(-1, -2) @ g @ y.transpose(-1, -2)

                # fp64 n = 9, 10: the ring of the smallest tile does not fit shared memory (DESIGN section 6 item 8)
                cases.append(Case(f"dense_inv_backward_{'sym_' if sym else ''}{t}_n{n}", dt, g_inv,
                                  lambda i, sym=sym: A.dense_inv_backward(i["y"], i["g"], sym), r_inv, rec=2, scale=10,
                                  extra=dict(strided=dt == torch.float64 and n >= 9)))
            # orders <= 3 closed-form cofactors on the tile kernel; from 4 pivoted, on the warp pool from 256 B of input
            cases.append(Case(f"dense_det_backward_{t}_n{n}", dt,
                              lambda b, s, n=n, dt=dt: dict(a=dense(b, n, dt, s), g=vecs(b, 1, dt, s + 1)[:, 0].contiguous()),
                              lambda i: A.dense_det_backward(i["a"], i["g"]),
                              lambda i: i["g"].double()[..., None, None] * torch.linalg.det(i["a"].double())[..., None, None]
                              * torch.linalg.inv(i["a"].double()).transpose(-1, -2), rec=2, scale=10,
                              extra=dict(path=3 if n >= 4 and (n * n + 1) * es >= 256 else 1)))
            for kk, rows, sym, sign in ((1, False, False, 1), (2, True, True, -1), (3, False, True, -1), (4, True, False, -1)):
                def g_out(b, s, n=n, dt=dt, kk=kk, rows=rows):
                    return dict(u=vecs(b, kk if rows else n, dt, s, k=n if rows else kk),
                                w=vecs(b, kk if rows else n, dt, s + 1, k=n if rows else kk))

                def r_out(i, rows=rows, sym=sym, sign=sign):
                    u, w = i["u"].double(), i["w"].double()
                    m = u.transpose(-1, -2) @ w if rows else u @ w.transpose(-1, -2)
                    return sign * ((m + m.transpose(-1, -2)) / 2 if sym else m)

                cases.append(Case(f"dense_outer_k{kk}_{'rows' if rows else 'left'}_{'sym' if sym else 'plain'}_"
                                  f"{'p' if sign > 0 else 'm'}_{t}_n{n}", dt, g_out,
                                  lambda i, rows=rows, sym=sym, sign=sign: A.dense_outer(i["u"], i["w"], rows, sym, sign),
                                  r_out, rec=2, scale=10, extra=dict(mag=True)))
            # A^-T B: one right-hand side (the one-row right division, many-right-hand-sides kernel), 2-4 (register
            # kernels with the transposed flag), more than 4 (the many-right-hand-sides kernel, transposed)
            for name, kk, right, algo in (("lu_k1", 1, False, _lib.ALGO_LU), ("lu_k3", 3, False, _lib.ALGO_LU),
                                          ("chol_k2", 2, False, _lib.ALGO_LDL), ("lu_right_k2", 2, True, _lib.ALGO_LU),
                                          ("lu_k5", 5, False, _lib.ALGO_LU)):
                def g_ts(b, s, n=n, dt=dt, kk=kk, right=right, algo=algo):
                    a = dense_spd(b, n, dt, s) if algo == _lib.ALGO_LDL else dense(b, n, dt, s)
                    return dict(a=a, b=vecs(b, kk, dt, s + 1, k=n) if right else vecs(b, n, dt, s + 1, k=kk))

                def r_ts(i, right=right):
                    a = i["a"].double()
                    if right:   # B A^-T = (A^-1 B^T)^T
                        return torch.linalg.solve(a, i["b"].double().transpose(-1, -2)).transpose(-1, -2)
                    return torch.linalg.solve(a.transpose(-1, -2), i["b"].double())

                cases.append(Case(f"tsolve_{name}_{t}_n{n}", dt, g_ts,
                                  lambda i, right=right, algo=algo: A.dense_tsolve(i["a"], i["b"], right, algo), r_ts,
                                  rec=2, scale=10, extra=dict(many=kk == 1 or kk > 4)))
            cases.append(Case(f"tmatvec_{t}_n{n}", dt, lambda b, s, n=n, dt=dt: dict(a=dense(b, n, dt, s), v=vecs(b, n, dt, s + 1)),
                              lambda i: A.dense_tmatvec(i["a"], i["v"]),
                              lambda i: (i["a"].double().transpose(-1, -2) @ i["v"].double()[..., None])[..., 0], scale=10))
            cases.append(Case(f"outer_backward_{t}_n{n}", dt,
                              lambda b, s, n=n, nn=nn, dt=dt: dict(x=vecs(b, n, dt, s), g=vecs(b, nn, dt, s + 1)),
                              lambda i: A.outer_backward(i["x"], i["g"]),
                              lambda i, n=n: 2 * (_ghat(i["g"], n) @ i["x"].double()[..., None])[..., 0], scale=10))
            cases.append(Case(f"to_full_backward_{t}_n{n}", dt, lambda b, s, n=n, dt=dt: dict(g=vecs(b, n, dt, s, k=n)),
                              lambda i: A.to_full_backward(i["g"]),
                              lambda i: _pack2(i["g"].double() + i["g"].double().transpose(-1, -2)) / 2, scale=10))
        for k, d in MATMUL_SHAPES:
            mode1 = k == d and k <= 3
            kh, ko = (d, k) if mode1 else (k, d)
            for which in (1, 2, 3):
                def g_mb(b, s, k=k, d=d, kh=kh, ko=ko, dt=dt):
                    j = 0.3 * vecs(b, k, dt, s, k=d) + 2 * torch.eye(k, d, device=DEV, dtype=dt)
                    return dict(j=j, h=spd(b, kh, dt, s + 1), g=vecs(b, ko * (ko + 1) // 2, dt, s + 2))

                def run_mb(i, which=which):
                    dj, dh = A.matmul_backward(i["j"], i["h"], i["g"], which)
                    return torch.cat([p for p in (None if dj is None else dj.flatten(-2), dh) if p is not None], -1)

                cases.append(Case(f"matmul_backward_w{which}_{t}_k{k}_d{d}", dt, g_mb, run_mb,
                                  lambda i, k=k, d=d, which=which: _matmul_backward(i, k, d, which), scale=10,
                                  extra=dict(mag=True)))
    return cases


_CASES = None


def all_cases():
    global _CASES
    if _CASES is None:
        _CASES = {c.name: c for c in _sym_cases() + _dense_cases() + _grad_cases()}
    return _CASES


# --------------------------------------------------------------------------
# planning from the launch record
# --------------------------------------------------------------------------

def _shape():
    from nitorch_fastmath_b200 import _lib
    return _lib.last_launch_shape()


def _path():
    from nitorch_fastmath_b200 import _lib
    return int(_lib.load().nfm_last_path_was_tma())


def _geom(sh):
    return tuple(sh[k] for k in ("kind", "threads", "mpt", "stages", "warps", "seg"))


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _call(case, batch, seed):
    ins = case.gen(batch, seed)
    out = case.run(ins)
    return ins, out, _shape(), _path()


def _unit(sh, batch):
    """Matrices per tile (tile kernel) or warp tile (pool, many right-hand sides)."""
    if sh["kind"] == 1:
        return sh["threads"] * sh["mpt"]
    if sh["kind"] == 4:
        return 32
    # pool: 32 matrices per warp tile, 16 when two lanes share a matrix
    return 16 if sh["tiles"] == -(-batch // 16) and sh["tiles"] != -(-batch // 32) else 32


def _need(sh, wraps):
    """Tiles (warp tiles) at which every CTA (warp) passes its ring `wraps` times."""
    if sh["kind"] == 1:
        return (wraps * sh["stages"] + 1) * sh["grid"]
    if sh["kind"] == 3:
        return (wraps + 1) * sh["stages"] * sh["grid"]
    return (wraps + 1) * sh["stages"] * sh["warps"] * sh["grid"]


def _wraps(sh):
    if sh["kind"] == 1:
        return (sh["tiles"] // sh["grid"] - 1) // sh["stages"]
    if sh["kind"] == 3:
        return (sh["tiles"] // sh["grid"] - 1) // sh["stages"]
    if sh["kind"] == 4:
        return (sh["tiles"] // (sh["grid"] * sh["warps"]) - 1) // sh["stages"]
    return 0


def _ragged(tiles, unit):
    """A batch of `tiles` tiles whose last one is partial, plus 3 matrices past the granule."""
    return (tiles - 1) * unit + unit // 2 + 3


def _grid_max_probe(case, sh0, batch0):
    """Grid of a launch with more tiles than resident CTAs."""
    unit = _unit(sh0, batch0)
    per_sm = 4 if sh0["kind"] == 4 else max(1, 2048 // sh0["threads"])
    tiles = _sms() * per_sm * max(1, sh0["warps"] if sh0["kind"] == 4 else 1) + 1
    b = _ragged(tiles, unit)
    _, _, sh, _ = _call(case, b, 7)
    return sh, b


def _bytes(ins, out):
    return sum(t.numel() * t.element_size() for t in ins.values()) + out.numel() * out.element_size()


def plan(case):
    """[(label, batch, launch record)] for the small geometry and, where the op has one, the large."""
    ins, out, sh0, path = _call(case, 4099, 3)
    if sh0["kind"] == 0:
        return [("none", 4099, sh0)]
    sh, b = _grid_max_probe(case, sh0, 4099)
    assert _geom(sh) == _geom(sh0), (case.name, sh0, sh)
    unit = _unit(sh, b)
    small = None
    for w in (2, 1):
        bs = _ragged(_need(sh, w), unit)
        _, o, shs, _ = _call(case, bs, 5)
        if _geom(shs) == _geom(sh0):
            small = (f"small/w{w}" if w == 1 else "small", bs, shs)
            break
    assert small is not None, f"{case.name}: the first geometry cannot pass its ring once"
    out = [small]
    if sh0["kind"] != 1:
        return out
    # double until the geometry switches (or no light op could still be below the switch)
    b, switched = small[1], None
    while True:
        b = 2 * b
        i2, o2, sh2, _ = _call(case, b, 5)
        if _geom(sh2) != _geom(sh0):
            switched = sh2
            break
        if _bytes(i2, o2) > STOP_BYTES:
            break
        del i2, o2
    if switched is None:
        return out
    ul = _unit(switched, b)
    assert switched["tiles"] > switched["grid"]
    tiles = max(_need(switched, 2), -(-b // ul) + 1)
    out.append(("large", _ragged(tiles, ul), None))
    return out


# --------------------------------------------------------------------------
# checking
# --------------------------------------------------------------------------

def _rel(got, want, rec, addend=None):
    got = got.double()
    dims = tuple(range(-rec, 0))
    if rec == 0:
        return ((got - want).abs() / want.abs().clamp_min(1e-300)).max()
    num = (got - want).pow(2).sum(dims).sqrt()
    if addend is not None:
        a = addend.double()
        den = a.pow(2).sum(dims).sqrt() + (want - a).pow(2).sum(dims).sqrt()
    else:
        den = want.pow(2).sum(dims).sqrt()
    return (num / den.clamp_min(1e-300)).max()


def worst_error(case, ins, out):
    worst = torch.zeros((), device=DEV, dtype=torch.float64)
    batch = out.shape[0]
    for c in range(0, batch, CHUNK):
        sl = {k: v[c:c + CHUNK] for k, v in ins.items()}
        want = case.ref(sl)
        if case.extra.get("dot"):      # a sum of products: error relative to the sum of their magnitudes
            den = (sl["u"].double() * sl["w"].double()).abs().sum(-1, keepdim=True)
            err = ((out[c:c + CHUNK].double() - want).abs() / den.clamp_min(1e-300)).max()
        elif case.extra.get("mag"):    # sums of products of random signs: norm-wise, relative to the same
            # formula on the magnitudes of the inputs (a record whose entries all nearly cancel has no exact digits)
            den = case.ref({k: v.abs() for k, v in sl.items()})
            dims = tuple(range(-case.rec, 0))
            num = (out[c:c + CHUNK].double() - want).pow(2).sum(dims).sqrt()
            err = (num / den.pow(2).sum(dims).sqrt().clamp_min(1e-300)).max()
            del den
        else:
            err = _rel(out[c:c + CHUNK], want, case.rec, sl.get(case.addend) if case.addend else None)
        worst = torch.maximum(worst, err)
        del want
    return float(worst)


def oracle_slices(case, ins, out):
    if case.oracle is None:
        return
    from oracle import generators as Gen
    batch = out.shape[0]
    m = min(case.oracle_rows, batch)
    for start in (0, max(0, batch // 2 - m // 2), batch - m):
        sl = slice(start, start + m)
        want = case.oracle({k: v[sl].cpu() for k, v in ins.items()})
        err = Gen.rel_err(out[sl], want, case.rec)
        assert err <= TOL[case.dtype] * case.scale, f"{case.name} oracle slice at {start}: {err:.3e}"


def _dense_aligned(ins):
    return all(t.is_contiguous() and t.data_ptr() % 16 == 0 for t in ins.values())


def run_case(case):
    steps = plan(case)
    rows = []
    small_batch = None
    for label, batch, sh_expected in steps:
        ins, out, sh, path = _call(case, batch, 11)
        warp = case.extra.get("warp")
        if warp:
            assert path == 2 and sh["kind"] == 0, (case.name, path, sh)
        elif case.extra.get("strided"):
            assert path == 0 and sh["kind"] == 0, (case.name, path, sh)
        elif _dense_aligned(ins) and not (case.extra.get("many") and sh["kind"] == 0):
            # (the many-right-hand-sides kernel stages only when three warps' buffers fit shared memory)
            assert path != 0, f"{case.name} ({label}, batch {batch}) fell off the TMA path: {sh}"
            assert path == case.extra.get("path", path), (case.name, label, path, sh)
        if label.startswith("small"):
            small_batch = batch
            if sh_expected is not None and label != "none":
                assert _geom(sh) == _geom(sh_expected)
        if label != "none" and not warp and not case.extra.get("strided"):
            want_w = 1 if label.endswith("w1") else 2
            assert _wraps(sh) >= want_w, (case.name, label, sh)
            if sh["kind"] == 4:   # whole warp tiles; the < 32 systems after them go to the one-thread kernel
                assert sh["tiles"] == batch // 32
            else:
                assert sh["tiles"] == -(-(batch - 3) // _unit(sh, batch)), (sh, batch)
        err = worst_error(case, ins, out)
        assert err <= TOL[case.dtype] * case.scale, f"{case.name} ({label}, batch {batch}): worst rel err {err:.3e}"
        if label == "large":
            assert _geom(sh) != _geom(steps[0][2])
            # the same call cut into chunks that run in the small geometry: the same bits
            cs = small_batch // 32 * 32
            parts = []
            for c in range(0, batch, cs):
                parts.append(case.run({k: v[c:c + cs] for k, v in ins.items()}))
                if c == 0:
                    assert _geom(_shape()) == _geom(steps[0][2])
            assert torch.equal(out, torch.cat(parts)), f"{case.name}: large geometry differs from the small one"
            del parts
        if label == steps[-1][0]:
            oracle_slices(case, ins, out)
        rows.append(dict(case=case.name, geometry=label, batch=batch, **sh, wraps=_wraps(sh), path=path, err=err))
        del ins, out
    COVERAGE.extend(rows)
    return rows


def _ids():
    # names only: the table is built without a GPU (the collection runs on CPU machines too)
    return [c for c in all_cases()]


@pytest.mark.gpu
@pytest.mark.parametrize("name", _ids())
def test_steady_state(name):
    run_case(all_cases()[name])


@pytest.mark.gpu
def test_scaled_identity_addmatvec_order7_stays_on_the_tma_path():
    """fp32 7x7 scaled-identity addmatvec: the large geometry's ring with the addend
    staged does not fit the shared memory; the small geometry must take the batch."""
    nfm = _nfm()
    b = 6 << 20
    mat = vecs(b, 1, torch.float32, 1, positive=True)
    vec, inp = vecs(b, 7, torch.float32, 2), vecs(b, 7, torch.float32, 3)
    y = nfm.sym_addmatvec(inp, mat, vec)
    assert _path() == 1 and _shape()["kind"] == 1
    assert torch.equal(y, inp + mat * vec)


@pytest.mark.gpu
def test_more_than_2_31_elements():
    """fp32 3x3 packed solve on 360 M matrices (2.16 G elements in `mat`): every matrix
    checked by a float64 residual, the far end against the oracle; on the TMA path and
    on a view with a storage offset (the head peel)."""
    nfm = _nfm()
    b = 360_000_003
    mat = torch.empty(b + 1, 6, device=DEV, dtype=torch.float32)
    g = torch.Generator(device=DEV).manual_seed(31)
    for c in range(0, b + 1, 16 << 20):
        m = min(16 << 20, b + 1 - c)
        a = torch.randn(m, 3, 3, device=DEV, generator=g)
        full = a @ a.transpose(-1, -2)
        full.diagonal(0, -1, -2).add_(3)
        mat[c:c + m] = _pack(full)
    vec = torch.randn(b + 1, 3, device=DEV, generator=g)
    assert mat[1:].numel() > 2 ** 31
    for m, v in ((mat[:b], vec[:b]), (mat[1:], vec[1:])):
        x = nfm.sym_solve(m, v)
        assert _path() == 1
        worst = 0.0
        for c in range(0, b, 16 << 20):
            a = _unpack(m[c:c + (16 << 20)].double(), 3)
            r = (a @ x[c:c + (16 << 20)].double()[..., None])[..., 0] - v[c:c + (16 << 20)].double()
            worst = max(worst, float((r.norm(dim=-1) / v[c:c + (16 << 20)].double().norm(dim=-1).clamp_min(1e-30)).max()))
        assert worst < 2e-5, worst
        sl = slice(b - SLICE, b)
        from oracle import generators as Gen
        assert Gen.rel_err(x[sl], P.sym_solve(m[sl].cpu(), v[sl].cpu())) <= TOL[torch.float32]
        del x
    del mat, vec
    torch.cuda.empty_cache()


# --------------------------------------------------------------------------
# path switches, in a child process
# --------------------------------------------------------------------------

SWITCH_CASES = ["solve_S_auto_none_f32_n3", "invert_auto_f32_n6", "batchinv_f64_n4", "addmatvec_E_f32_n7",
                "batchinv_f64_n8", "batchinv_f64_n9", "batchinv_f64_n10", "solvevec_f32_n10",
                "lmdiv_lu_k5_f64_n4", "lmdiv_lu_k12_f32_n6", "rmdiv_k1_f64_n8",
                "dense_inv_backward_f32_n4", "matmul_backward_w3_f32_k6_d6", "tsolve_lu_k1_f64_n8"]


def _digest(t):
    return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()


def run_subset(jobs):
    """[(case, batch)] -> per job: output digest, worst error against float64, launch record, path."""
    res = []
    for name, batch in jobs:
        case = all_cases()[name]
        ins, out, sh, path = _call(case, batch, 11)
        res.append(dict(name=name, batch=batch, digest=_digest(out), err=worst_error(case, ins, out), path=path, **sh))
        del ins, out
    return res


def _child_main(argv):
    jobs, dest = json.loads(argv[0]), argv[1]
    res = run_subset(jobs)
    np.savez(dest, records=np.array(json.dumps(res)))
    torch.cuda.synchronize()


SWITCHES = [("NFM_DISABLE_PDL", "1"), ("NFM_BALANCE", "1"), ("NFM_MANY_TRANSPOSE_FROM", "64"),
            ("NFM_MANY_TRANSPOSE_FROM", "1"), ("NFM_DISABLE_PAIR_INVERSE", "1"), ("NFM_DISABLE_MANY_STAGED", "1")]


@pytest.fixture(scope="module")
def switch_jobs():
    """The subset at batches sized from its default launch record: tile cases in both
    geometries (a batch that equal-tile scheduling cuts), the pool and many-RHS kernels."""
    jobs = []
    for name in SWITCH_CASES:
        case = all_cases()[name]
        for label, batch, sh in plan(case):
            _, _, sh2, _ = _call(case, batch, 11)
            if sh2["kind"] == 1:
                unit = _unit(sh2, batch)
                batch = _ragged(max(sh2["grid"] + 1, int(0.9 * sh2["tiles"])), unit)
            jobs.append((name, batch))
    return jobs, run_subset(jobs)


@pytest.mark.gpu
@pytest.mark.parametrize("var,value", SWITCHES)
def test_path_switch_in_a_child_process(tmp_path, switch_jobs, var, value):
    jobs, base = switch_jobs
    dest = str(tmp_path / "child.npz")
    env = dict(os.environ, **{var: value})
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    code = "import sys, test_steady_state as T; T._child_main(sys.argv[1:])"
    r = subprocess.run([sys.executable, "-c", code, json.dumps(jobs), dest], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    child = json.loads(str(np.load(dest)["records"]))
    assert [c["name"] for c in child] == [b["name"] for b in base]
    cut = set()
    for b, c in zip(base, child):
        case = all_cases()[b["name"]]
        assert c["err"] <= TOL[case.dtype] * case.scale, (var, c)
        if var in ("NFM_DISABLE_PDL", "NFM_BALANCE", "NFM_MANY_TRANSPOSE_FROM"):
            assert c["digest"] == b["digest"], (var, value, b["name"], b["batch"])
        if var == "NFM_BALANCE" and c["kind"] == 1:
            if c["tiles"] > -(-c["batch"] // (c["threads"] * c["mpt"])):
                cut.add((c["threads"], c["mpt"], c["stages"]))
        if var == "NFM_DISABLE_PAIR_INVERSE" and b["name"].startswith("batchinv_f64_n") and int(b["name"][14:]) >= 8:
            assert b["tiles"] == -(-b["batch"] // 16) and c["tiles"] == -(-c["batch"] // 32), (b, c)
        if var == "NFM_DISABLE_MANY_STAGED" and b["kind"] == 4:
            assert c["path"] == 0 and c["kind"] == 0, c
        if var == "NFM_MANY_TRANSPOSE_FROM" and c["kind"] == 4:
            # slot 5 of the record is the re-layout mask: 64 never re-lays a tile out, 1 always the matrices
            assert (c["seg"] == 0) if value == "64" else (c["seg"] & 1) == 1, (value, c)
    if var == "NFM_BALANCE":
        geoms = {(b["threads"], b["mpt"], b["stages"]) for b in base if b["kind"] == 1}
        # equal tiles cut a launch of a few waves; large launches keep the full capacity by design
        # (balanced_tile: the rounding to kTileGran absorbs the cut), so only the small geometries must show it
        assert len(cut) >= 1 and cut <= geoms, (cut, geoms)


def teardown_module(module):
    if not COVERAGE:
        return
    lines = [f"{'case':40s} {'geometry':9s} {'batch':>10s} {'thr':>4s} {'mpt':>3s} {'st':>3s} {'warps':>5s} {'seg':>3s} "
             f"{'grid':>5s} {'tiles':>8s} {'wraps':>5s} {'worst err':>9s}"]
    for r in COVERAGE:
        lines.append(f"{r['case']:40s} {r['geometry']:9s} {r['batch']:10d} {r['threads']:4d} {r['mpt']:3d} {r['stages']:3d} "
                     f"{r['warps']:5d} {r['seg']:3d} {r['grid']:5d} {r['tiles']:8d} {r['wraps']:5d} {r['err']:9.2e}")
    lines.append(f"peak device memory: {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    path = os.environ.get("NFM_COVERAGE_TABLE")
    if path:
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")
    print("\n" + "\n".join(lines))
