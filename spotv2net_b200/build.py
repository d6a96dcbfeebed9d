"""In-tree build of libspotv2_gat.so (sm_100a only, plain nvcc, no ATen/pybind).

``python -m spotv2net_b200.build`` or ``__graft_entry__.build()``.  The .so is
git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OBJ = PKG / "_build"
LIB = PKG / "libspotv2_gat.so"

SOURCES = ["api.cu", "fold.cu", "gemm_simt.cu", "gemm_tc.cu", "gemm_f16.cu", "proj.cu", "attn_fwd.cu", "attn_fwd16.cu", "attn_prep.cu", "attn_bwd.cu", "attn_bwd2.cu", "attn_bwd3.cu", "attn_large.cu", "windows.cu", "edge_grad.cu"]
# SPOTV2_BRINGUP=1 in the environment compiles the cycle counters of the attention kernels (tools/fwd16_waits.py,
# tools/fwd_waits.py) and the GEMM's timing probe in; the product build carries none of them
NVCC_FLAGS = (["-DSPOTV2_BRINGUP"] if os.environ.get("SPOTV2_BRINGUP") else []) + [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libspotv2_gat.so cannot be built")


def _digest(path: Path) -> str:
    h = hashlib.sha256()
    for dep in sorted(list(CSRC.glob("*.cuh")) + [path, PKG.parent / "include" / "spotv2_gat.h"]):
        h.update(dep.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile(src: str, verbose: bool) -> Path:
    path = CSRC / src
    obj = OBJ / (src + ".o")
    stamp = OBJ / (src + ".sha")
    dig = _digest(path)
    if obj.exists() and stamp.exists() and stamp.read_text() == dig:
        return obj
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", str(path), "-o", str(obj)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    (OBJ / (src + ".log")).write_text(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{res.stdout}\n{res.stderr}")
    if verbose:
        sys.stderr.write(res.stderr)
    stamp.write_text(dig)
    return obj


def build(verbose: bool = False, force: bool = False) -> Path:
    OBJ.mkdir(exist_ok=True)
    if force:
        for f in OBJ.glob("*.sha"):
            f.unlink()
    sources = [s for s in SOURCES if (CSRC / s).exists()]
    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), sources))
    newest = max(o.stat().st_mtime for o in objs)
    if force or not LIB.exists() or LIB.stat().st_mtime < newest:
        cmd = [_nvcc(), "-shared", "-o", str(LIB), *map(str, objs), "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
