"""Builds libb200rt.so (CUDA kernels + C ABI) in-tree for sm_100a.

    python -m cpp_raytracer_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  -fmad=false is REQUIRED for parity: the FP64 primitive
tests must not be contracted into FMAs (the reference is built for baseline x86-64, which has
none), see csrc/traverse.cuh.  Places that want an FMA call __fmaf_rn explicitly.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200rt.so")
SOURCES = ["api.cu", "kernels.cu", "wavefront.cu", "lbvh.cu", "scene_layout.cu", "devmem.cu", "bvh_builder.cpp"]
HEADERS = ["bvh_builder.h", "devmem.h", "kernels.h", "thread_pool.h", "traverse.cuh", "shade.cuh", "path.cuh", "rng.cuh",
           os.path.join("..", "..", "include", "b200rt.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
    "-ccbin", "g++",
    "-Xcompiler", "-fPIC,-pthread,-ffp-contract=off,-O3",
    "-Xptxas", "-v",
    "-shared",
]


HOST_DIR = os.path.join(HERE, "host")
HOST_BIN = os.path.join(HOST_DIR, "b200rt_scenes")
HOST_DEPS = ["scenes_main.cpp", "scenes.hpp", os.path.join("include", "b200rt", "raytracer.hpp")]


def build_host(force: bool = False) -> str:
    """Builds host/b200rt_scenes: the reference's scene set written against the API-compatible
    C++ headers (host/include), linked against libb200rt.so."""
    deps = [os.path.join(HOST_DIR, d) for d in HOST_DEPS] + [LIB]
    if not force and os.path.exists(HOST_BIN) and all(os.path.getmtime(d) <= os.path.getmtime(HOST_BIN) for d in deps):
        return HOST_BIN
    cmd = ["g++", "-std=c++20", "-O2", "-ffp-contract=off", "-I" + os.path.join(HOST_DIR, "include"),
           "-o", HOST_BIN, os.path.join(HOST_DIR, "scenes_main.cpp"), "-L" + HERE, "-lb200rt", "-Wl,-rpath,$ORIGIN/.."]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("g++ failed building host/b200rt_scenes")
    return HOST_BIN


FLAGS_STAMP = os.path.join(HERE, "build.flags")


def _extra_flags() -> list:
    return os.environ.get("B200RT_NVCC_EXTRA", "").split()   # experiment knob, e.g. -DB200RT_PATH_MINB=12


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    # a library built with other experiment flags than the ones asked for now is stale too
    built_with = open(FLAGS_STAMP).read().split() if os.path.exists(FLAGS_STAMP) else []
    if built_with != _extra_flags():
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


LIB_DBG = os.path.join(HERE, "libb200rt_dbg.so")


def build_debug(force: bool = False) -> str:
    """libb200rt_dbg.so: the same sources with -DB200RT_DEBUG_BOUNDS (every traversal-stack push, node / primitive /
    material index and frame store range-checked on the device; b200rt_debug_bounds reports the counts).  The GPU
    suite renders every scene through it (tests/test_gpu_bounds.py): the stand-in for compute-sanitizer, which
    the GPU pool does not allow."""
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    if not force and os.path.exists(LIB_DBG) and all(os.path.getmtime(d) <= os.path.getmtime(LIB_DBG) for d in deps if os.path.exists(d)):
        return LIB_DBG
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in NVCC_FLAGS if f not in ("-Xptxas", "-v")]
    cmd = [nvcc, *flags, "-DB200RT_DEBUG_BOUNDS", "-o", LIB_DBG, *[os.path.join(CSRC, s) for s in SOURCES], "-lpthread"]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libb200rt_dbg.so")
    return LIB_DBG


def build_variant(name: str, extra_flags: list) -> str:
    """An experiment build of the same sources with extra -D flags -> scratch_libs/libb200rt_<name>.so (git-ignored,
    travels to the GPU box; select it with B200RT_LIB).  For A/B measurements in one gpurun call."""
    out_dir = os.path.join(os.path.dirname(HERE), "scratch_libs")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, f"libb200rt_{name}.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-o", out, *[os.path.join(CSRC, s) for s in SOURCES], "-lpthread"]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    with open(out + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError(f"nvcc failed building {out}")
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = _extra_flags()
    cmd = [nvcc, *NVCC_FLAGS, *extra, "-o", LIB, *[os.path.join(CSRC, s) for s in SOURCES], "-lpthread"]
    env = dict(os.environ)
    env.pop("CXX", None)   # this image exports a CXX wrapper without libgomp specs
    env.pop("CC", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    log = res.stdout + res.stderr
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if verbose or res.returncode != 0:
        sys.stderr.write(log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libb200rt.so (see cpp_raytracer_b200/build.log)")
    with open(FLAGS_STAMP, "w") as f:
        f.write(" ".join(extra))
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, verbose=a.verbose))
    print(build_host(force=a.force))
    print(build_debug(force=a.force))
