"""Build libamplisolve_b200.so (CUDA kernels + C ABI + host code) in-tree for sm_100a.

    python -m amplisolve_b200.build [--force]

nvcc cross-compiles without a GPU.  -fmad=false: the reference runs on x86-64 without FMA and the
parity-critical fp32/fp64 expressions must not be contracted (they also use explicit _rn intrinsics).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "lib" / "libamplisolve_b200.so"
BIN = PKG / "bin"
OBJ = PKG / "lib" / "obj"
CU_SOURCES = ["as_kernels.cu", "as_noise_pattern.cu", "as_call_deferred.cu", "as_capi.cu", "as_sort.cu", "as_fisher.cu", "as_pileup.cu", "as_sites.cu"]
CXX_SOURCES = ["as_host.cpp", "as_bam.cpp", "as_serve.cpp"]  # as_bam.cpp inflates BGZF blocks with zlib (-lz)
HEADERS = ["as_device.cuh", "as_noise.cuh", "as_pipeline.cuh", "as_call.cuh", "as_kernels.h", "as_wire.h", "as_bam.h",
           "../../include/amplisolve_b200.h"]
# -cudart shared: the CUDA runtime is NOT linked into the product library (a static runtime would carry every runtime entry
# point, used or not, into libamplisolve_b200.so); libcudart.so.12 comes from the toolkit (rpath) or from the process
# (torch loads its own copy first in bench.py / the tests -- every runtime symbol this library imports exists there).
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC,-O2,-ffp-contract=off", "-cudart", "shared"]
CUDA_LIB_DIRS = ["/usr/local/cuda/lib64"]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(exe).exists():
        raise RuntimeError("nvcc not found: libamplisolve_b200.so cannot be built (there is no CPU fallback)")
    return exe


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def _compile(src: Path, obj: Path, verbose: bool):
    cmd = [nvcc(), *NVCC_FLAGS, "-c", "-o", str(obj), str(src), "-I", str(ROOT / "include")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, r


def check_no_batch_memcpy(paths) -> None:
    """The shipped binaries must not carry the batched-memcpy entry points of the CUDA runtime (they would only be there
    through a statically linked runtime: this library copies with plain cudaMemcpyAsync / cudaMemcpy2DAsync)."""
    import re
    pat = re.compile(rb"Memcpy(3D)?BatchAsync")
    for p in paths:
        if Path(p).exists() and pat.search(Path(p).read_bytes()):
            raise RuntimeError(f"{p} contains a batched-memcpy runtime symbol: link the CUDA runtime dynamically (-cudart shared)")


def build(force: bool = False, verbose: bool = False) -> Path:
    from concurrent.futures import ThreadPoolExecutor
    srcs = [CSRC / s for s in CU_SOURCES + CXX_SOURCES]
    hdrs = [CSRC / h for h in HEADERS] + [Path(__file__)]
    OBJ.mkdir(parents=True, exist_ok=True)
    jobs = []
    for src in srcs:
        obj = OBJ / (src.stem + ".o")
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as pool:
            for src, r in pool.map(lambda j: _compile(j[0], j[1], verbose), jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(f"== {src.name}\n" + r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed compiling {src.name}")
    objs = [OBJ / (src.stem + ".o") for src in srcs]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc(), *NVCC_FLAGS, "-shared", "-o", str(LIB), *map(str, objs), "-lz"]
        for d in CUDA_LIB_DIRS:
            cmd += ["-Xlinker", f"-rpath={d}"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed linking libamplisolve_b200.so")
    check_no_batch_memcpy([LIB])
    mains = CSRC / "as_main.cpp"
    if mains.exists():
        BIN.mkdir(exist_ok=True)
        for prog, macro in (("AmpliSolveErrorEstimation", "AS_MAIN_EE"), ("AmpliSolveVariantCalling", "AS_MAIN_VC"),
                            ("computeCounts", "AS_MAIN_CC"), ("amplisolve_b200_serve", "AS_MAIN_SERVE")):
            out = BIN / prog
            if force or _stale(out, [mains, LIB]):
                cmd = ["g++", "-O2", "-std=c++17", f"-D{macro}", "-o", str(out), str(mains), "-I", str(ROOT / "include"),
                       f"-L{LIB.parent}", "-lamplisolve_b200", "-Wl,-rpath,$ORIGIN/../lib"]
                r = subprocess.run(cmd, capture_output=True, text=True)
                if r.returncode != 0:
                    sys.stderr.write(r.stdout + r.stderr)
                    raise RuntimeError(f"g++ failed building {prog}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
