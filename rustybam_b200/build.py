"""Builds the in-tree native artefacts: librbcuda.so (CUDA, sm_100a) and the C++ host tools.

    python -m rustybam_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.path.join(HERE, "librbcuda.so")
RB = os.path.join(HERE, "rb")
HOSTLIB = os.path.join(HERE, "librbhost.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-Wall", "-Xptxas", "-v"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources(d, exts):
    return sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith(exts)) if os.path.isdir(d) else []


def build_cuda(force=False, verbose=False):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    srcs = _sources(CSRC, (".cu",))
    deps = srcs + _sources(CSRC, (".cuh", ".hpp")) + [os.path.join(ROOT, "include", "rbcuda.h"), os.path.abspath(__file__)]
    if not force and not _newer(LIB, deps):
        return LIB
    extra = os.environ.get("RB_NVCC_DEFS", "").split()  # e.g. "-DRB_LIFT_THREADS=256 -DRB_LIFT_MINB=2" (tuning sweeps)
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-shared", "-o", LIB] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building librbcuda.so")
    with open(os.path.join(HERE, "_build_ptxas.log"), "w") as f:
        f.write(r.stdout + r.stderr)
    return LIB


def build_host(force=False, verbose=False):
    """C++ host side: PAF/BED text loaders, synthetic generator, and the `rb` CLI (links librbcuda.so)."""
    srcs = _sources(HOST, (".cpp",))
    if not srcs:
        return None
    deps = srcs + _sources(HOST, (".hpp", ".h")) + [os.path.join(ROOT, "include", "rbcuda.h"), os.path.abspath(__file__),
                                                    os.path.join(CSRC, "f32_fmt.cuh"), os.path.join(CSRC, "rb_common.cuh"),  # (f32_fast.hpp includes them)
                                                    os.path.join(CSRC, "name_intern.hpp")]
    gxx = shutil.which("g++") or "g++"
    common = ["-O2", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread", "-I", os.path.join(ROOT, "include"), "-I", HOST]
    lib_srcs = [s for s in srcs if not s.endswith("rb_main.cpp")]
    if force or _newer(HOSTLIB, deps):
        r = subprocess.run([gxx] + common + ["-shared", "-o", HOSTLIB] + lib_srcs + ["-lz"], capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("g++ failed building librbhost.so")
    main = os.path.join(HOST, "rb_main.cpp")
    if os.path.exists(main) and (force or _newer(RB, deps + [LIB])):
        cmd = [gxx] + common + ["-o", RB, main] + lib_srcs + ["-L", HERE, "-lrbcuda", "-Wl,-rpath,$ORIGIN", "-lz"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("g++ failed building rb")
    return HOSTLIB


def build_all(force=False, verbose=False):
    build_cuda(force, verbose)
    build_host(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
    print("built", LIB)
