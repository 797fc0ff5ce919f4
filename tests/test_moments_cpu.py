"""CPU tests of the second-moment feature: the variance helper, the new C ABI entry without a device, and the host-layer
program of tests/test_gpu_moments.py (Camera::render_with_noise / render_to_noise) compiling and linking."""
import ctypes
import os

import numpy as np
import pytest


def test_sample_variance_matches_numpy():
    from cpp_raytracer_b200 import capi
    rng = np.random.default_rng(3)
    for n in (2, 3, 17, 256):
        x = rng.gamma(0.5, 4.0, size=(n, 5, 4, 3))          # skewed, like path-traced radiance
        mean = x.mean(axis=0)
        m2 = (x * x).mean(axis=0)
        got = capi.sample_variance(mean, m2, n)
        assert got.dtype == np.float64 and got.shape == mean.shape
        assert np.allclose(got, np.var(x, axis=0, ddof=1), rtol=1e-9, atol=1e-12)
    # all samples equal: rounding can put m2 a hair below mean^2; the result is clamped at 0
    mean = np.full(4, 0.7, np.float32)
    assert (capi.sample_variance(mean, mean.astype(np.float64) ** 2 * (1 - 1e-7), 8) == 0).all()
    # one sample gives no variance estimate
    one = capi.sample_variance(np.ones((2, 3)), np.ones((2, 3)), 1)
    assert one.shape == (2, 3) and np.isinf(one).all()


def test_render_moments_without_a_scene_is_einval():
    from cpp_raytracer_b200 import capi
    out = np.zeros(3, np.float32)
    m2 = np.zeros(3, np.float32)
    cam = np.zeros(1, capi.CAMERA_DTYPE)
    cam["image_w"] = 1; cam["image_h"] = 1; cam["spp"] = 1
    opts = capi.RenderOpts(0, 0, 0, 0, 0)
    lib = capi.lib()
    assert lib.b200rt_render_moments(None, cam.ctypes.data, ctypes.byref(opts), out.ctypes.data, m2.ctypes.data, None) == capi.EINVAL
    assert lib.b200rt_render_moments(None, cam.ctypes.data, ctypes.byref(opts), out.ctypes.data, None, None) == capi.EINVAL
    assert lib.b200rt_render_moments(None, None, None, None, None, None) == capi.EINVAL


def test_noise_program_compiles(tmp_path):
    """The host-layer program of the GPU suite builds here without a GPU."""
    from test_gpu_moments import compile_program
    assert os.path.exists(compile_program(tmp_path))
