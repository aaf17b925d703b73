"""Build the C-ABI shared library (libmmrs_b200.so) in-tree with nvcc for sm_100a.

The library is linked against the static CUDA runtime so that it loads on a machine without a
GPU or driver (the symbol-export test runs there); anything that needs the driver
(cuTensorMapEncodeTiled) is resolved at run time through cudaGetDriverEntryPoint.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_DIR = PKG_DIR / "lib"
LIB_PATH = LIB_DIR / "libmmrs_b200.so"
SOURCES = ["api.cu", "scan_gemv.cu", "scan_mma.cu", "select.cu", "selfjoin.cu", "selfjoin_mma.cu", "range.cu",
           "dedup_resolve.cu"]
HEADERS = ["common.cuh", "plan.h", "tcgen05_utils.cuh"]
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the mmrs_b200 CUDA library cannot be built")


def _stale(target: Path, deps: list[Path]) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every .cu to an object and link libmmrs_b200.so; returns its path."""
    nvcc = _nvcc()
    LIB_DIR.mkdir(exist_ok=True)
    obj_dir = PKG_DIR / "build"
    obj_dir.mkdir(exist_ok=True)
    hdrs = [CSRC / h for h in HEADERS] + [PKG_DIR.parent / "include" / "mmrs_b200.h"]
    common = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
              "--expt-relaxed-constexpr", "-DMMRS_BUILD"] + ARCH_FLAGS
    if verbose:
        common += ["-Xptxas", "-v"]
    objs = []
    procs = []
    for src in SOURCES:
        s = CSRC / src
        o = obj_dir / (src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc, "-c", str(s), "-o", str(o)] + common
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"nvcc failed on {src}:\n{out}\n")
        elif verbose and out:
            sys.stderr.write(f"--- {src}\n{out}\n")
    if failed:
        raise RuntimeError("nvcc compilation failed")
    if force or procs or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", str(LIB_PATH)] + [str(o) for o in objs] + ARCH_FLAGS + ["-cudart", "static"]
        subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
