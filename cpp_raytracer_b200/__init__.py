"""cpp_raytracer_b200 -- B200-native (sm_100a CUDA) implementation of cpp_raytracer's
per-pixel-sample path-tracing loop, behind the C ABI of include/b200rt.h.

Layout:
    csrc/         CUDA kernels, host BVH builder and the C ABI  -> libb200rt.so (built in-tree)
    capi.py       ctypes marshalling of the C ABI (no compute, no fallback)
    scene_io.py   flat scene / ray file formats shared with the oracle bridge
    host/         API-compatible C++ headers (Scene, Sphere, Camera::render ...) over the C ABI
    dist.py       sample-split multi-GPU render + NCCL reduce (one process per GPU)
"""
from .capi import (B200rtError, DeviceSceneHandle, HostScene, camera_init, camera_with, device_count,  # noqa: F401
                   lib, render_scene, sample_variance, selftest_bvh, tonemap)
from .scene_io import load_scene, save_scene  # noqa: F401

__all__ = ["B200rtError", "DeviceSceneHandle", "HostScene", "camera_init", "camera_with", "device_count",
           "lib", "render_scene", "sample_variance", "selftest_bvh", "tonemap", "load_scene", "save_scene"]
