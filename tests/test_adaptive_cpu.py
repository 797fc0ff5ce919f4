"""CPU tests of adaptive sampling: the C entry without a scene, the host-side replay of the convergence rule the GPU suite
relies on, and the host-layer program of tests/test_gpu_adaptive.py (Camera::render_adaptive) compiling and linking."""
import ctypes
import os

import numpy as np


def test_render_adaptive_without_a_scene_is_einval():
    from cpp_raytracer_b200 import capi
    out = np.zeros(3, np.float32)
    cam = np.zeros(1, capi.CAMERA_DTYPE)
    cam["image_w"] = 1; cam["image_h"] = 1; cam["spp"] = 4
    opts = capi.RenderOpts(0, 0, 0, 0, 0)
    aopts = capi.AdaptiveOpts(2, 2, 0.1, 0.0)
    lib = capi.lib()
    assert lib.b200rt_render_adaptive(None, cam.ctypes.data, ctypes.byref(opts), ctypes.byref(aopts), out.ctypes.data,
                                      None, None, None) == capi.EINVAL
    assert lib.b200rt_render_adaptive(None, None, None, None, None, None, None, None) == capi.EINVAL


def test_replay_follows_the_rule():
    """The replay on synthetic planes: a flat pixel is converged, a noisy one is not, and the 3 x 3 dilation keeps the
    neighbours of a noisy pixel going while the rest stop after the first pass."""
    from test_gpu_adaptive import converged, dilate, pass_counts, replay
    assert pass_counts(6, 12, 42) == [6, 18, 30, 42]
    assert pass_counts(32, 8, 24) == [24]
    h, w = 7, 9
    flat = np.full((h, w, 3), 0.5, np.float32)
    uni = {n: (flat, flat * flat) for n in pass_counts(4, 4, 16)}
    assert converged(flat, flat * flat, 4, 0.0, 0.0).all()
    noisy_m2 = (flat * flat).copy()
    noisy_m2[3, 4] = 1.0                        # one pixel with variance
    uni = {n: (flat, noisy_m2) for n in pass_counts(4, 4, 16)}
    assert not converged(flat, noisy_m2, 4, 0.01, 0.0)[3, 4]
    spp = replay(uni, 4, 4, 16, 0.01, 0.0)
    want = np.where(dilate(np.pad(np.ones((1, 1), bool), ((3, h - 4), (4, w - 5)))), 16, 4)
    assert np.array_equal(spp, want)


def test_adaptive_program_compiles(tmp_path):
    """The host-layer program of the GPU suite builds here without a GPU."""
    from test_gpu_adaptive import compile_program
    assert os.path.exists(compile_program(tmp_path))
