"""Build recipe for libvoitta_b200.so (nvcc, sm_100a only) — used by __graft_entry__.build()."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
SRC = HERE / "csrc" / "vb_api.cu"
LIB = HERE / "libvoitta_b200.so"
FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-Xcompiler", "-fPIC", "-shared"]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; libvoitta_b200.so cannot be built")
    return p


def needs_build(lib: Path | None = None) -> bool:
    lib = lib or LIB
    if not lib.exists():
        return True
    t = lib.stat().st_mtime
    srcs = list((HERE / "csrc").glob("*")) + [HERE.parent / "include" / "voitta_b200.h"]
    return any(s.stat().st_mtime > t for s in srcs)


LIB_DEBUG = HERE / "libvoitta_b200_dbg.so"


def build_debug() -> Path:
    """The same library with -DVB_DEBUG_BOUNDS: every VB_CHECK becomes a device-side assert (tools/gpu_sanitize.sh;
    select it with VB200_LIB=<path>).  compute-sanitizer is closed on the GPU pool; these are our own bounds checks."""
    cmd = [nvcc_path(), *FLAGS, "-DVB_DEBUG_BOUNDS", "-o", str(LIB_DEBUG), str(SRC)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{r.stdout}\n{r.stderr}")
    return LIB_DEBUG


def build(force: bool = False, verbose: bool = False, debug: bool = True) -> Path:
    """Release library and (debug=True) the bounds-checked one, each only when older than its sources; the two nvcc
    runs go side by side.  A stale debug library once made tools/gpu_sanitize.sh test yesterday's kernels."""
    jobs = []
    if force or needs_build(LIB):
        cmd = [nvcc_path(), *FLAGS, "-o", str(LIB), str(SRC)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        jobs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    if debug and (force or needs_build(LIB_DEBUG)):
        jobs.append(subprocess.Popen([nvcc_path(), *FLAGS, "-DVB_DEBUG_BOUNDS", "-o", str(LIB_DEBUG), str(SRC)],
                                     stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for j in jobs:
        out, err = j.communicate()
        if j.returncode != 0:
            raise RuntimeError(f"nvcc failed:\n{out}\n{err}")
        if verbose:
            print(err)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
