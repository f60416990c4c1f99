"""Builds libdgod_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

The library has no torch dependency: it is plain CUDA behind `include/dgod_b200.h`.  The built
`.so` lives next to this file so that it travels with the repo snapshot to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
OBJ_DIR = PKG_DIR / "build"
LIB_PATH = PKG_DIR / "libdgod_b200.so"
SOURCES = ["error.cu", "tmap.cu", "match.cu", "fcos.cu", "fcos_loss.cu", "fcos_post.cu", "sampler.cu", "nms.cu", "rpn.cu", "roi_align.cu",
           "roi_align_fast.cu", "roi_align_tma.cu", "roi_align_own.cu", "misc.cu", "transform.cu",
           "fpn.cu", "bottleneck.cu", "map_eval.cu", "linear_tc.cu", "rpn_head.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    # The bit-exact kernels use __f*_rn intrinsics (never contracted); -fmad=false additionally
    # keeps the compiler from fusing anything else, matching the CPU reference's arithmetic.
    "-fmad=false",
    "-Xptxas", "-v",
]
# DGOD_DEBUG_WAITS=1: bounded mbarrier waits in the tcgen05 kernels (a lost arrive is reported instead of hanging).
if os.environ.get("DGOD_DEBUG_WAITS"):
    NVCC_FLAGS.append("-DDGOD_DEBUG_WAITS")


def _nvcc() -> str:
    cand = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    return cand if Path(cand).exists() else "nvcc"


def _stale(target: Path, deps: list[Path]) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every .cu under csrc/ and link libdgod_b200.so.  Returns the library path."""
    OBJ_DIR.mkdir(exist_ok=True)
    headers = sorted(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "dgod_b200.h"]
    jobs = []
    for name in SOURCES:
        src = CSRC / name
        obj = OBJ_DIR / (src.stem + ".o")
        if force or _stale(obj, [src] + headers):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", str(src), "-o", str(obj)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        (OBJ_DIR / (src.stem + ".ptxas.log")).write_text(res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            print(res.stderr, file=sys.stderr)
        return obj

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [OBJ_DIR / (Path(s).stem + ".o") for s in SOURCES]
    if force or jobs or _stale(LIB_PATH, objs):
        cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a",
               "-o", str(LIB_PATH), *map(str, objs)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    return LIB_PATH


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
