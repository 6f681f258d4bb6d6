"""Builds the reference (facebookresearch/Pearl, pure Python) for the tests of the plugin boundary with it: every module of
its `pearl` package is byte-compiled into oracle/_ref/pearl/ as a sourceless .pyc, which Python imports directly, so
oracle/_ref/ on sys.path makes `pearl` importable (test infrastructure; oracle/_ref/ is git-ignored).  The checkout is
taken from $PEARL_REFERENCE_ROOT, else /root/reference, the location the golden fixtures were recorded from
(oracle/gen_golden.py); where neither exists nothing is built and those tests skip."""
from __future__ import annotations

import os
import py_compile
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def reference_root() -> str | None:
    for root in (os.environ.get("PEARL_REFERENCE_ROOT", ""), "/root/reference"):
        if root and os.path.isdir(os.path.join(root, "pearl")):
            return root
    return None


def build() -> str | None:
    """Returns the directory to put on sys.path, or None when the reference is not on this machine."""
    root = reference_root()
    if root is None:
        return None
    shutil.rmtree(OUT, ignore_errors=True)
    for dirpath, dirnames, files in os.walk(os.path.join(root, "pearl")):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        rel = os.path.relpath(dirpath, root)
        for f in files:
            if f.endswith(".py"):
                py_compile.compile(os.path.join(dirpath, f), cfile=os.path.join(OUT, rel, f[:-3] + ".pyc"),
                                   dfile=os.path.join(rel, f), doraise=True)
    return OUT
