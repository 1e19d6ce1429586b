"""In-tree build of the native libraries (explicit nvcc / g++ command lines, no JIT cache).

  librt_b200.so       CUDA core for sm_100a, exports exactly include/rt_b200.h
  librt_b200_host.so  C++ host mirror of the reference crate's interface + its C shim
                      (include/rt_b200_host.h); links against librt_b200.so

`python -m rs_pathtracing_b200.build` builds both (nvcc cross-compiles without a GPU).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
CORE_SO = os.path.join(HERE, "librt_b200.so")
HOST_SO = os.path.join(HERE, "librt_b200_host.so")

CORE_SOURCES = [os.path.join(CSRC, f) for f in ("rt_core.cu", "rt_march_kernels.cu")]
OBJ_DIR = os.path.join(HERE, "build")
CORE_HEADERS = [
    os.path.join(CSRC, "rt_queues.cuh"),
    os.path.join(CSRC, "rt_math.cuh"),
    os.path.join(CSRC, "rt_scene.cuh"),
    os.path.join(CSRC, "rt_march.cuh"),
    os.path.join(CSRC, "rt_cull.cuh"),
    os.path.join(CSRC, "march_bounds.hpp"),
    os.path.join(ROOT, "include", "rt_b200.h"),
]
HOST_SOURCES = [os.path.join(CSRC, "host", "ray_tracing.cpp"), os.path.join(CSRC, "host", "host_c.cpp")]
HOST_HEADERS = [
    os.path.join(CSRC, "host", "ray_tracing.hpp"),
    os.path.join(CSRC, "host", "json.hpp"),
    os.path.join(ROOT, "include", "rt_b200_host.h"),
    os.path.join(ROOT, "include", "rt_b200.h"),
]

# -fmad=false: the parity contract forbids contracting a*b+c (the reference is plain Rust f64);
# explicit fma() calls in the culling code are unaffected.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math",
    "-Xptxas", "-v",
    "-diag-suppress", "20014",   # surface_func_t<Jet2> is a host-only instantiation of a __host__ __device__ template
]
NVCC_LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static"]
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-shared"]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd: list[str], log_name: str | None = None) -> None:
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if log_name:
        with open(os.path.join(HERE, log_name), "w") as f:
            f.write(" ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd))


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def build_core(force: bool = False) -> str:
    """one object per translation unit, compiled in parallel (no relocatable device code: every kernel is launched
    from its own unit), then linked into librt_b200.so"""
    deps = CORE_HEADERS + [os.path.abspath(__file__)]
    extra = os.environ.get("RT_B200_NVCC_EXTRA", "").split()   # tuning experiments, e.g. -DRT_MARCH_MIN_BLOCKS=3
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs, jobs = [], []
    for src in CORE_SOURCES:
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or extra or _stale(obj, [src] + deps):
            log = "build_" + os.path.basename(src)[:-3] + ".log"
            jobs.append((threading.Thread(target=_run_job, args=([nvcc_path(), *NVCC_FLAGS, *extra, "-c", "-o", obj, src], log)),
                         obj))
    errors = []
    for t, _ in jobs:
        t.start()
    for t, obj in jobs:
        t.join()
    errors = [e for e in _JOB_ERRORS]
    _JOB_ERRORS.clear()
    if errors:
        raise RuntimeError("build failed:\n" + "\n".join(errors))
    if jobs or not os.path.exists(CORE_SO) or _stale(CORE_SO, objs):
        _run([nvcc_path(), *NVCC_LINK_FLAGS, "-o", CORE_SO, *objs])
        # one log with every unit's ptxas -v output (registers / spills), as before
        with open(os.path.join(HERE, "build_core.log"), "w") as out:
            for src in CORE_SOURCES:
                lp = os.path.join(HERE, "build_" + os.path.basename(src)[:-3] + ".log")
                if os.path.exists(lp):
                    out.write(open(lp).read())
    return CORE_SO


_JOB_ERRORS: list[str] = []


def _run_job(cmd: list[str], log_name: str) -> None:
    try:
        _run(cmd, log_name)
    except Exception as e:   # collected by build_core
        _JOB_ERRORS.append(str(e))


def build_host(force: bool = False) -> str:
    build_core(force)
    if force or _stale(HOST_SO, HOST_SOURCES + HOST_HEADERS + [CORE_SO, os.path.abspath(__file__)]):
        cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
        _run([cxx, *CXX_FLAGS, "-o", HOST_SO, *HOST_SOURCES, "-L" + HERE, "-lrt_b200", "-Wl,-rpath,$ORIGIN"])
    return HOST_SO


def build_all(force: bool = False) -> None:
    build_core(force)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
    print(CORE_SO)
    print(HOST_SO)
