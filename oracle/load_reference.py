"""Import the *real*, unmodified reference: from the directory that the
environment variable NFM_REFERENCE_ROOT names, else from the git-ignored
install ``baseline/_ref/`` that ``oracle/install_reference.py`` makes.  The
reference is not part of this repository; without it the callers fall back to
the stored fixtures in ``tests/golden/`` or to the pinned port.

TEST / MEASUREMENT INFRASTRUCTURE ONLY -- used by
``oracle/validate_against_reference.py``, ``tests/golden/make_golden.py`` and
the reference arm of ``bench.py`` (``--impl reference``).  Nothing under
nitorch_fastmath_b200/ imports it.

``import nitorch_fastmath`` needs the un-vendored ``jitfields`` package
(sym.py:37, tests/utils.py:2).  Following SURVEY.md appendix A.6 we load
``_impl/sym.py`` by path (it only needs torch), register an in-memory
``jitfields`` whose ``sym`` sub-module binds the nine public names of
``sym.py:30-34`` to that file, and then import the package normally.
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import sys
import types
import warnings

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_root() -> str:
    env = os.environ.get("NFM_REFERENCE_ROOT")
    local = os.path.join(_REPO, "baseline", "_ref")
    for root in ([env] if env else []) + [local]:
        if os.path.isfile(os.path.join(root, "nitorch_fastmath", "_impl", "sym.py")):
            return root
    return env or local


REFERENCE_ROOT = _find_root()


def available() -> bool:
    return os.path.isfile(
        os.path.join(REFERENCE_ROOT, "nitorch_fastmath", "_impl", "sym.py"))


def load():
    """Returns (ref_sym_impl, ref_batched_impl, ref_sugar) modules."""
    if not available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    import torch

    warnings.filterwarnings("ignore")
    path = os.path.join(REFERENCE_ROOT, "nitorch_fastmath", "_impl", "sym.py")
    spec = importlib.util.spec_from_file_location("_nfm_ref_sym_impl", path)
    ref_sym = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_sym)

    if "jitfields" not in sys.modules:
        jf = types.ModuleType("jitfields")
        jf.set_num_threads = torch.set_num_threads
        jfs = types.ModuleType("jitfields.sym")
        jfs.sym_matvec = ref_sym.sym_matvec
        jfs.sym_solve = ref_sym.sym_solve
        jfs.sym_invert = ref_sym.sym_invert
        jfs.sym_addmatvec = lambda i, m, v: i + ref_sym.sym_matvec(m, v)
        jfs.sym_submatvec = lambda i, m, v: i - ref_sym.sym_matvec(m, v)
        jfs.sym_addmatvec_ = lambda i, m, v: i.add_(ref_sym.sym_matvec(m, v))
        jfs.sym_submatvec_ = lambda i, m, v: i.sub_(ref_sym.sym_matvec(m, v))
        jfs.sym_solve_ = lambda m, v, *a: v.copy_(ref_sym.sym_solve(m, v, *a))
        jfs.sym_invert_ = lambda m: m.copy_(ref_sym.sym_invert(m))
        jfs.__all__ = [k for k in vars(jfs) if k.startswith("sym_")]
        jf.sym = jfs
        sys.modules["jitfields"] = jf
        sys.modules["jitfields.sym"] = jfs
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    ref_batched = importlib.import_module("nitorch_fastmath._impl.batched")
    ref_sugar = importlib.import_module("nitorch_fastmath.sugar")
    return ref_sym, ref_batched, ref_sugar
