"""In-tree nvcc build of libbhsparse_b200.so (sm_100a only).

`python -m benchmark_spgemm_using_csr_b200.build [--force] [--verbose]`

One object per translation unit (compiled in parallel), linked into
benchmark_spgemm_using_csr_b200/lib/libbhsparse_b200.so.  The .so is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "lib", "obj")
LIB = os.path.join(HERE, "lib", "libbhsparse_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = [
    "context.cu",
    "stage_count.cu",
    "stage_small.cu",
    "stage_symbolic.cu",
    "stage_range.cu",
    "stage_pattern.cu",
    "pattern_plan.cu",
    "direct_plan.cu",
    "dist_nccl.cu",
    "stage_bucket.cu",
    "stage_numeric_f32.cu",
    "stage_numeric_f64.cu",
    "stage_numeric_none.cu",
    "stage_numeric_c64.cu",
    "stage_numeric_c128.cu",
    "stage_transpose.cu",
    "stage_masked.cu",
]
HEADERS = ["common.cuh", "stage_numeric.cuh", "stage_range.cuh", "stage_range_vec.cuh", "stage_pattern.cuh", "pattern_plan.h", "direct_plan.h", "context.h", "stage_bucket.cuh", os.path.join(INCLUDE, "bhsparse_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-I", INCLUDE,
]


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def ccbin() -> list[str]:
    """nvcc's host compiler: the image's $CC wrapper lacks some specs; use the system g++"""
    return ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []


def _newest_header() -> float:
    t = 0.0
    for h in HEADERS:
        p = h if os.path.isabs(h) else os.path.join(CSRC, h)
        t = max(t, os.path.getmtime(p))
    return t


def _stale(out: str, src: str, hdr_time: float) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return t < os.path.getmtime(src) or t < hdr_time


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    cc = nvcc()
    hdr_time = _newest_header()
    extra = ["-Xptxas", "-v"] if verbose else []

    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, src, hdr_time):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [cc] + ccbin() + NVCC_FLAGS + extra + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return job, r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for (src, obj), r in ex.map(compile_one, jobs):
                if verbose and (r.stdout or r.stderr):
                    sys.stderr.write(r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if jobs or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [cc] + ccbin() + ["-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


DRIVER_SRC = os.path.join(os.path.dirname(HERE), "examples", "spgemm_driver.cpp")
DRIVER_BIN = os.path.join(os.path.dirname(HERE), "examples", "spgemm")


def build_driver(force: bool = False) -> str:
    """The reference-compatible CLI driver (examples/spgemm_driver.cpp) on top of
    include/bhsparse.h: `examples/spgemm -cuda -spgemm <0..4|A.mtx> [B.mtx]`."""
    lib = build()
    hdrs = [os.path.join(INCLUDE, "bhsparse.h"), os.path.join(INCLUDE, "bhsparse_b200.h"), DRIVER_SRC]
    if (not force and os.path.exists(DRIVER_BIN)
            and all(os.path.getmtime(DRIVER_BIN) >= os.path.getmtime(h) for h in hdrs)):
        return DRIVER_BIN
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else (shutil.which("g++") or "g++")
    cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-I", INCLUDE, DRIVER_SRC, "-o", DRIVER_BIN,
           "-L", os.path.dirname(lib), "-lbhsparse_b200", "-Wl,-rpath,$ORIGIN/../benchmark_spgemm_using_csr_b200/lib"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"driver build failed:\n{r.stdout}\n{r.stderr}")
    return DRIVER_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
    if "--driver" in sys.argv:
        print(build_driver(force=True))
