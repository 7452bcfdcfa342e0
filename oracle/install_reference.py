#!/usr/bin/env python
"""Installs the UNMODIFIED reference hot-path package into oracle/_ref/ (git-ignored), compiled to bytecode.

`pip install` of habitat-lab cannot work here: its setup pulls gym, omegaconf, hydra-core, habitat_sim ... which are not
installed, and the package `__init__`s import them.  The hot-path modules themselves only need torch / numpy, so the
install byte-compiles every `habitat_baselines` python module into a sourceless `.pyc` at the place the source has in
the reference tree; oracle/ref_shim.py imports them with arithmetic-free stubs for the absent third-party packages.
`__graft_entry__.build()` runs this when the reference checkout is readable (`HB200_REFERENCE_SRC`, else
`reference_path` in BASELINE.json); oracle/_ref then goes wherever the built tree goes.  Nothing under oracle/_ref is
product code: only `bench.py --impl reference`, the `torch_cuda_baseline` leg of bench.py and tests use it."""
import json
import os
import py_compile
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
PKG = os.path.join("habitat-baselines", "habitat_baselines")


def reference_src() -> str:
    env = os.environ.get("HB200_REFERENCE_SRC")
    if env:
        return env
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


def install(verbose=True) -> bool:
    ref = reference_src()
    src = os.path.join(ref, PKG)
    if not os.path.isdir(src):
        return False
    dst = os.path.join(DST, PKG)
    n = 0
    for dirpath, dirnames, files in os.walk(src):
        dirnames[:] = [d for d in dirnames if d not in ("__pycache__", "config")]
        for f in files:
            if not f.endswith(".py"):
                continue
            s = os.path.join(dirpath, f)
            rel = os.path.relpath(s, src)
            d = os.path.join(dst, rel + "c")
            if not os.path.exists(d) or os.path.getmtime(d) < os.path.getmtime(s):
                os.makedirs(os.path.dirname(d), exist_ok=True)
                py_compile.compile(s, cfile=d, dfile=os.path.join(PKG, rel), doraise=True)
            n += 1
    lic = os.path.join(ref, "LICENSE")
    if os.path.exists(lic):
        shutil.copyfile(lic, os.path.join(DST, "LICENSE"))
    if verbose:
        print(f"reference: {n} modules of {PKG} compiled into {dst}")
    return True


if __name__ == "__main__":
    if not install():   # not an error: the reference arms and tests then run without it (see their docstrings)
        print(f"reference: {os.path.join(reference_src(), PKG)} not readable, oracle/_ref not installed", file=sys.stderr)
