"""Build libkissmcmc_cuda.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libkissmcmc_cuda.so"
SOURCES = ["kmc_api.cu", "kmc_aux.cu", "kmc_metro.cu", "kmc_ops_exp.cu", "kmc_ops_gauss.cu", "kmc_ops_misc.cu",
           "kmc_ops_mix.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; libkissmcmc_cuda.so cannot be built")


def _stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "kissmcmc_cuda.h"]
    return any(p.stat().st_mtime > t for p in deps)


def build_library(force: bool = False, verbose: bool = False, out: Path | None = None, defines=()) -> Path:
    """Compile every translation unit (in parallel) and link libkissmcmc_cuda.so.  `out` / `defines` build a variant
    (e.g. build/variants/x.so with -DKMC_PUSH_THREADS=128) without touching the in-tree library."""
    from concurrent.futures import ThreadPoolExecutor
    lib = Path(out) if out else LIB
    if not force and not out and not _stale():
        return LIB
    ccbin = os.environ.get("CXX") or shutil.which("g++") or "/usr/bin/g++"      # host compiler: $CXX, else g++ on PATH
    objdir = PKG.parent / "build" / ("obj_" + lib.stem)
    objdir.mkdir(parents=True, exist_ok=True)

    def compile_one(src):
        obj = objdir / (Path(src).stem + ".o")
        cmd = [_nvcc(), *NVCC_FLAGS, *defines, "-ccbin", ccbin, "-c", "-o", str(obj), str(CSRC / src)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        res = list(ex.map(compile_one, SOURCES))
    if verbose:
        print("".join(e for _, e in res))
    lib.parent.mkdir(parents=True, exist_ok=True)
    r = subprocess.run([_nvcc(), *LINK_FLAGS, "-ccbin", ccbin, "-o", str(lib), *[str(o) for o, _ in res]],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return lib


if __name__ == "__main__":
    import sys
    if len(sys.argv) > 1:      # python build.py <out.so> [-DNAME=VALUE ...]: a variant build
        print(build_library(force=True, verbose=True, out=Path(sys.argv[1]), defines=sys.argv[2:]))
    else:
        print(build_library(force=True, verbose=True))
