"""Builds libdsp_lp.so (the C-ABI of include/dsp_lp.h) in-tree for sm_100a with nvcc.

    python -m dispatches_b200.csrc.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
LIB = HERE / "libdsp_lp.so"
SOURCES = [HERE / "dsp_lp.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", f"-I{ROOT / 'include'}"]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: cannot build libdsp_lp.so")
    return p


def needs_build():
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = SOURCES + [ROOT / "include" / "dsp_lp.h"] + sorted(HERE.glob("*.cuh"))
    return any(s.stat().st_mtime > t for s in deps)


def build(force=False, verbose=False):
    """Builds the library if sources are newer.  Serialised across processes with a file lock: under torchrun every rank
    calls this at start-up and only the first one may run nvcc.  An up-to-date library is returned without writing
    anything, so that a built tree can be used read-only."""
    import fcntl
    if not force and not needs_build():
        return LIB
    with open(HERE / ".build.lock", "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lk, fcntl.LOCK_UN)


def _build_locked(force, verbose):
    if not force and not needs_build():
        return LIB
    cmd = [nvcc_path(), *NVCC_FLAGS, *(["-Xptxas", "-v"] if verbose else []), *map(str, SOURCES), "-o", str(LIB)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
