#!/usr/bin/env python
"""Install the UNMODIFIED reference into the git-ignored ``baseline/_ref/`` so that
``bench.py --impl reference`` can time the reference's own code and
``tests/test_oracle.py`` can compare the port with it bit for bit.

TEST / MEASUREMENT INFRASTRUCTURE ONLY -- nothing under nitorch_fastmath_b200/
imports it.  Needs a checkout of nitorch-fastmath, named by NFM_REFERENCE_SRC:

    NFM_REFERENCE_SRC=<nitorch-fastmath checkout> python oracle/install_reference.py

Steps (outcome recorded in baseline/_ref/INSTALL_LOG.txt and DESIGN.md section 7):
 1. ``pip install --no-index --no-build-isolation --no-deps --target baseline/_ref``
    from a scratch copy of the checkout (which may be read-only).
 2. The reference's setup.py lists ``packages=['nitorch_fastmath']`` only, so the
    wheel omits the ``_impl`` (and ``tests``) sub-packages that ``batched.py`` and
    ``sugar.py`` import: the installed tree is completed by copying those
    directories verbatim from the checkout.  Nothing is edited.
The un-vendored dependency ``jitfields`` is not installable offline; the loader
(oracle/load_reference.py) registers an in-memory stand-in that binds the nine
names of ``nitorch_fastmath/sym.py:30-34`` to the reference's own ``_impl/sym.py``.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("NFM_REFERENCE_SRC", "")
DST = os.path.join(ROOT, "baseline", "_ref")


def main() -> int:
    if not os.path.isdir(os.path.join(SRC, "nitorch_fastmath")):
        print(f"NFM_REFERENCE_SRC={SRC!r} holds no nitorch_fastmath package: keeping whatever baseline/_ref holds")
        return 0
    shutil.rmtree(DST, ignore_errors=True)
    os.makedirs(DST, exist_ok=True)
    log = []
    with tempfile.TemporaryDirectory() as tmp:
        work = os.path.join(tmp, "reference")
        shutil.copytree(SRC, work)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--target", DST, work]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        log.append("$ " + " ".join(cmd))
        log.append(r.stdout[-2000:])
        log.append(f"pip exit code {r.returncode}")
    pkg = os.path.join(DST, "nitorch_fastmath")
    if r.returncode != 0 or not os.path.isdir(pkg):
        shutil.copytree(os.path.join(SRC, "nitorch_fastmath"), pkg, dirs_exist_ok=True)
        log.append("pip install failed: copied the package directory verbatim instead")
    for sub in ("_impl", "tests"):
        if not os.path.isdir(os.path.join(pkg, sub)):
            shutil.copytree(os.path.join(SRC, "nitorch_fastmath", sub), os.path.join(pkg, sub))
            log.append(f"wheel omitted sub-package {sub!r} (setup.py packages=['nitorch_fastmath']): copied verbatim")
    with open(os.path.join(DST, "INSTALL_LOG.txt"), "w") as f:
        f.write("\n".join(log) + "\n")
    print("\n".join(log[-4:]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
