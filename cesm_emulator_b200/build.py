"""Build libcesm_b200.so (hand-written sm_100a kernels + the C ABI) in-tree with nvcc.

The shared library is git-ignored but travels with the working tree to the GPU box, so it is
built here (nvcc cross-compiles without a GPU) and only rebuilt when a source is newer.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
BUILD_DIR = PKG_DIR / "csrc" / "build"
LIB_PATH = PKG_DIR / "libcesm_b200.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _newest_header_mtime() -> float:
    hs = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "cesm_b200.h"]
    return max(h.stat().st_mtime for h in hs if h.exists())


def build(force: bool = False, verbose: bool = False) -> Path:
    sources = sorted(CSRC.glob("*.cu"))
    if not sources:
        raise RuntimeError(f"no CUDA sources under {CSRC}")
    BUILD_DIR.mkdir(parents=True, exist_ok=True)
    hdr_mtime = _newest_header_mtime()
    nvcc = _nvcc()

    def compile_one(src: Path):
        obj = BUILD_DIR / (src.stem + ".o")
        if (not force and obj.exists() and obj.stat().st_mtime >= src.stat().st_mtime
                and obj.stat().st_mtime >= hdr_mtime):
            return obj, None
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
        (BUILD_DIR / (src.stem + ".ptxas.log")).write_text(r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, len(sources))) as ex:
        results = list(ex.map(compile_one, sources))
    objs = [o for o, _ in results]
    rebuilt = any(log is not None for _, log in results)
    if verbose:
        for _, log in results:
            if log:
                sys.stderr.write(log)
    if rebuilt or force or not LIB_PATH.exists():
        cmd = [nvcc, "-shared", "-o", str(LIB_PATH), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB_PATH


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose=True)
    print(p)
