"""Build libraglite_b200.so in-tree with nvcc for sm_100a (no torch extension machinery: the library
is a plain C-ABI shared object, see include/raglite_b200.h)."""

from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB_DIR = PKG / "lib"
LIB_PATH = LIB_DIR / "libraglite_b200.so"

NVCC_FLAGS = [
    "-shared", "-Xcompiler", "-fPIC", "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a", "--expt-extended-lambda",
]


def _nvcc() -> str | None:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    return None


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def is_stale() -> bool:
    if not LIB_PATH.exists():
        return True
    lib_m = LIB_PATH.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "raglite_b200.h"]
    return any(p.stat().st_mtime > lib_m for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA source into ``raglite_b200/lib/libraglite_b200.so`` (sm_100a only)."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libraglite_b200.so")
    LIB_DIR.mkdir(exist_ok=True)
    # One process per GPU: every rank may find the library stale at the same moment.  An exclusive file
    # lock serialises them (the first one builds, the others re-check and find it fresh), and the output
    # goes to a per-process temporary that is renamed into place, so nobody ever loads a half-written .so.
    import fcntl

    with open(LIB_DIR / ".build.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale():
                return LIB_PATH
            tmp = LIB_PATH.with_suffix(f".so.tmp{os.getpid()}")
            extra = os.environ.get("RL_NVCC_EXTRA", "").split()   # extra nvcc flags (e.g. -Xptxas=-warn-spills)
            cmd = [nvcc, *NVCC_FLAGS, *extra, "-o", str(tmp), *[str(s) for s in sources()]]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            proc = subprocess.run(cmd, capture_output=True, text=True, check=False)
            if proc.returncode != 0:
                tmp.unlink(missing_ok=True)
                raise RuntimeError(f"nvcc failed:\n{proc.stdout}\n{proc.stderr}")
            if verbose:
                print(proc.stderr)
            tmp.replace(LIB_PATH)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH
