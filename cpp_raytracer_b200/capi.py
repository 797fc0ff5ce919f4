"""ctypes binding of include/b200rt.h (libb200rt.so, built in-tree by cpp_raytracer_b200.build).

The library is the product; this module only marshals numpy buffers into it.  There is no
Python or CPU fallback anywhere: if the shared library is missing the import fails loudly, and
if there is no CUDA device every compute call raises B200rtError(ENODEVICE).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# B200RT_LIB selects another build of the same library (the bounds-checked libb200rt_dbg.so the GPU suite runs
# in place of compute-sanitizer); it must export the same ABI.
LIB_PATH = os.environ.get("B200RT_LIB") or os.path.join(HERE, "libb200rt.so")

# ---- struct dtypes (must mirror include/b200rt.h; checked against sizeof in tests) ---------
MATERIAL_DTYPE = np.dtype([("kind", "<u4"), ("pad", "<u4"), ("rgb", "<f8", 3), ("param", "<f8")])
SPHERE_DTYPE = np.dtype([("c", "<f8", 3), ("r", "<f8"), ("mat", "<u4"), ("prim", "<u4")])
QUAD_DTYPE = np.dtype([("v", "<f8", 3), ("s1", "<f8", 3), ("s2", "<f8", 3), ("mat", "<u4"), ("prim", "<u4")])
CAMERA_DTYPE = np.dtype([
    ("image_w", "<u8"), ("image_h", "<u8"), ("spp", "<u8"), ("max_depth", "<u8"),
    ("center", "<f8", 3), ("dir", "<f8", 3), ("up", "<f8", 3),
    ("focus_dist", "<f8"), ("defocus_angle", "<f8"), ("vfov", "<f8"), ("hfov", "<f8"),
    ("background", "<f8", 3),
    ("pixel00", "<f8", 3), ("delta_x", "<f8", 3), ("delta_y", "<f8", 3), ("disk_x", "<f8", 3), ("disk_y", "<f8", 3),
])
assert MATERIAL_DTYPE.itemsize == 40 and SPHERE_DTYPE.itemsize == 40 and QUAD_DTYPE.itemsize == 80

MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC, MAT_LIGHT = 0, 1, 2, 3
VARIANT_MEGAKERNEL, VARIANT_WAVEFRONT = 0, 1
FLAG_SUM, FLAG_ACCUMULATE, FLAG_COUNTERS, FLAG_EXACT_COUNT, FLAG_THREAD_PIXELS = 1, 2, 4, 8, 16
BUILDER_AUTO, BUILDER_HOST_SAH, BUILDER_GPU_LBVH = 0, 1, 2
OK, EINVAL, ENODEVICE, ECUDA, ENOMEM, EINTERNAL = 0, -1, -2, -3, -4, -5


class SceneDesc(C.Structure):
    _fields_ = [("n_materials", C.c_uint64), ("n_spheres", C.c_uint64), ("n_quads", C.c_uint64),
                ("materials", C.c_void_p), ("spheres", C.c_void_p), ("quads", C.c_void_p)]


class BuildOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_leaf_prims", C.c_int32), ("sah_bins", C.c_int32),
                ("build_threads", C.c_int32), ("builder", C.c_int32)]


class SceneInfo(C.Structure):
    _fields_ = [("n_prims", C.c_uint64), ("n_spheres", C.c_uint64), ("n_quads", C.c_uint64),
                ("n_materials", C.c_uint64), ("n_nodes", C.c_uint64), ("device_bytes", C.c_uint64),
                ("tree_depth", C.c_uint32), ("stack_entries", C.c_uint32),
                ("build_ms", C.c_double), ("upload_ms", C.c_double), ("n_hoisted", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RenderOpts(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("sample_offset", C.c_uint64), ("sample_count", C.c_uint64),
                ("variant", C.c_int32), ("flags", C.c_uint32)]


class AdaptiveOpts(C.Structure):
    _fields_ = [("min_spp", C.c_uint32), ("step_spp", C.c_uint32), ("rel_noise", C.c_double), ("abs_noise", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double), ("total_ms", C.c_double),
                ("paths", C.c_uint64), ("rays", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("build_ms", C.c_double), ("replicate_ms", C.c_double), ("exchange_ms", C.c_double),
                ("n_devices", C.c_uint32), ("peer_exchange", C.c_uint32), ("quad_tests", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/b200rt.h declares; tests check the library exports exactly these
SHADE_RECORD_DTYPE = np.dtype([("scattered", "<f8", 6), ("t", "<f8"), ("atten", "<f4", 3), ("emit", "<f4", 3),
                               ("prim", "<i4"), ("flags", "<i4")])
assert SHADE_RECORD_DTYPE.itemsize == 88

EXPORTS = {
    "b200rt_device_count": (C.c_int, []),
    "b200rt_last_error": (C.c_char_p, []),
    "b200rt_version": (C.c_int, []),
    "b200rt_trim": (C.c_int, []),
    "b200rt_scene_create": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(BuildOpts), C.POINTER(C.c_void_p)]),
    "b200rt_scene_create_multi": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(BuildOpts), C.POINTER(C.c_int32), C.c_int32,
                                            C.POINTER(C.c_void_p)]),
    "b200rt_render_scene_multi": (C.c_int, [C.POINTER(SceneDesc), C.c_void_p, C.POINTER(RenderOpts), C.POINTER(BuildOpts),
                                            C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.POINTER(Stats), C.POINTER(SceneInfo)]),
    "b200rt_debug_philox": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int]),
    "b200rt_debug_samplers": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]),
    "b200rt_debug_bounds": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200rt_scene_info": (C.c_int, [C.c_void_p, C.POINTER(SceneInfo)]),
    "b200rt_scene_destroy": (None, [C.c_void_p]),
    "b200rt_camera_init": (C.c_int, [C.c_void_p]),
    "b200rt_raycast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "b200rt_render": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RenderOpts), C.c_void_p, C.POINTER(Stats)]),
    "b200rt_render_device": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RenderOpts), C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "b200rt_render_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RenderOpts), C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "b200rt_render_adaptive": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RenderOpts), C.POINTER(AdaptiveOpts), C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "b200rt_render_scene": (C.c_int, [C.POINTER(SceneDesc), C.c_void_p, C.POINTER(RenderOpts), C.POINTER(BuildOpts),
                                      C.c_void_p, C.POINTER(Stats), C.POINTER(SceneInfo)]),
    "b200rt_tonemap": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int]),
    "b200rt_tonemap_device": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "b200rt_debug_camera_rays": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int]),
    "b200rt_debug_shade": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_void_p]),
    "b200rt_debug_lane_accounting": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RenderOpts), C.c_void_p]),
    "b200rt_finalize_device": (C.c_int, [C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "b200rt_finalize_peers_device": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int64, C.c_double, C.c_void_p,
                                               C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "b200rt_selftest_bvh": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(BuildOpts), C.POINTER(SceneInfo)]),
}


class B200rtError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libb200rt error {code}: {message}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """Loads libb200rt.so; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m cpp_raytracer_b200.build` "
                "(there is no CPU/Python fallback for the render path)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def _check(rc: int):
    if rc != 0:
        raise B200rtError(rc, lib().b200rt_last_error().decode(errors="replace"))


def device_count() -> int:
    return lib().b200rt_device_count()


@dataclass
class HostScene:
    """Flat host-side scene: the numpy mirror of B200rtSceneDesc (+ the scene's camera)."""
    materials: np.ndarray
    spheres: np.ndarray
    quads: np.ndarray
    camera: np.ndarray   # 0-d CAMERA_DTYPE record array (shape (1,))
    name: str = ""

    @property
    def n_prims(self) -> int:
        return len(self.spheres) + len(self.quads)

    def desc(self) -> SceneDesc:
        self.materials = np.ascontiguousarray(self.materials, dtype=MATERIAL_DTYPE)
        self.spheres = np.ascontiguousarray(self.spheres, dtype=SPHERE_DTYPE)
        self.quads = np.ascontiguousarray(self.quads, dtype=QUAD_DTYPE)
        return SceneDesc(len(self.materials), len(self.spheres), len(self.quads),
                         self.materials.ctypes.data, self.spheres.ctypes.data, self.quads.ctypes.data)


def camera_init(cam: np.ndarray) -> np.ndarray:
    """Camera::init() (reference camera.h:87-157) on a copy of `cam`; returns the copy."""
    out = np.array(cam, dtype=CAMERA_DTYPE).reshape(1).copy()
    _check(lib().b200rt_camera_init(out.ctypes.data))
    return out


def camera_with(cam: np.ndarray, **kw) -> np.ndarray:
    """Copy of `cam` with fields overridden (image_w, image_h, spp, max_depth ...) and the
    derived block recomputed."""
    out = np.array(cam, dtype=CAMERA_DTYPE).reshape(1).copy()
    for k, v in kw.items():
        out[k] = v
    return camera_init(out)


def selftest_bvh(scene: HostScene, max_leaf_prims: int = 0, sah_bins: int = 0, threads: int = 0) -> dict:
    info = SceneInfo()
    desc = scene.desc()
    bo = BuildOpts(-1, max_leaf_prims, sah_bins, threads, 0)
    _check(lib().b200rt_selftest_bvh(C.byref(desc), C.byref(bo), C.byref(info)))
    return info.as_dict()


class DeviceSceneHandle:
    """Owns a b200rt scene handle (device-resident scene + BVH)."""

    def __init__(self, scene: HostScene, device: int = -1, max_leaf_prims: int = 0, sah_bins: int = 0, threads: int = 0,
                 builder: int = BUILDER_AUTO, devices=None):
        """`devices`: a list of CUDA ordinals makes the scene resident on all of them (b200rt_scene_create_multi:
        built once on devices[0], copied to the others); render() then splits the samples across them."""
        self._h = C.c_void_p()
        desc = scene.desc()
        if devices is not None:
            devs = (C.c_int32 * len(devices))(*[int(d) for d in devices])
            bo = BuildOpts(int(devices[0]) if len(devices) else -1, max_leaf_prims, sah_bins, threads, builder)
            _check(lib().b200rt_scene_create_multi(C.byref(desc), C.byref(bo), devs, len(devices), C.byref(self._h)))
        else:
            bo = BuildOpts(device, max_leaf_prims, sah_bins, threads, builder)
            _check(lib().b200rt_scene_create(C.byref(desc), C.byref(bo), C.byref(self._h)))
        self.host = scene

    def close(self):
        if self._h:
            lib().b200rt_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def info(self) -> dict:
        info = SceneInfo()
        _check(lib().b200rt_scene_info(self._h, C.byref(info)))
        return info.as_dict()

    def raycast(self, rays: np.ndarray, tmin: float = 1e-5, tmax: float = float("inf")):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        prim = np.empty(n, dtype=np.int32)
        t = np.empty(n, dtype=np.float64)
        _check(lib().b200rt_raycast(self._h, rays.ctypes.data, n, tmin, tmax, prim.ctypes.data, t.ctypes.data))
        return prim, t

    def debug_shade(self, rays: np.ndarray, rnd: np.ndarray, tmin: float = 1e-5, tmax: float = float("inf")) -> np.ndarray:
        """One surface interaction per ray with caller-supplied random words (b200rt_debug_shade);
        returns a record array of SHADE_RECORD_DTYPE."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        rnd = np.ascontiguousarray(rnd, dtype=np.uint32).reshape(-1, 4)
        if rnd.shape[0] != rays.shape[0]:
            raise ValueError("one row of four random words per ray")
        out = np.zeros(rays.shape[0], dtype=SHADE_RECORD_DTYPE)
        _check(lib().b200rt_debug_shade(self._h, rays.ctypes.data, rnd.ctypes.data, rays.shape[0], tmin, tmax, out.ctypes.data))
        return out

    def render(self, cam: np.ndarray, seed: int = 0xB200, sample_offset: int = 0, sample_count: int = 0,
               variant: int = VARIANT_MEGAKERNEL, flags: int = 0):
        cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
        h, w = int(cam["image_h"][0]), int(cam["image_w"][0])
        out = np.empty((h, w, 3), dtype=np.float32)
        opts = RenderOpts(seed, sample_offset, sample_count, variant, flags)
        st = Stats()
        _check(lib().b200rt_render(self._h, cam.ctypes.data, C.byref(opts), out.ctypes.data, C.byref(st)))
        return out, st.as_dict()

    def render_moments(self, cam: np.ndarray, seed: int = 0xB200, sample_offset: int = 0, sample_count: int = 0, flags: int = 0):
        """render() plus each pixel's second moment (b200rt_render_moments): returns (mean, m2, stats), where m2 is the
        mean over the samples of x^2 per channel (both planes are sums with FLAG_SUM).  sample_variance(mean, m2, n) turns
        them into the per-pixel sample variance.  Default kernel only: the wavefront variant, FLAG_THREAD_PIXELS and
        FLAG_COUNTERS are EINVAL."""
        cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
        h, w = int(cam["image_h"][0]), int(cam["image_w"][0])
        mean = np.empty((h, w, 3), dtype=np.float32)
        m2 = np.empty((h, w, 3), dtype=np.float32)
        opts = RenderOpts(seed, sample_offset, sample_count, VARIANT_MEGAKERNEL, flags)
        st = Stats()
        _check(lib().b200rt_render_moments(self._h, cam.ctypes.data, C.byref(opts), mean.ctypes.data, m2.ctypes.data, C.byref(st)))
        return mean, m2, st.as_dict()

    def render_adaptive(self, cam: np.ndarray, rel_noise: float, abs_noise: float = 0.0, min_spp: int = 16, step_spp: int = 16,
                        seed: int = 0xB200, sample_offset: int = 0, sample_count: int = 0, flags: int = 0):
        """Adaptive sampling (b200rt_render_adaptive): each pixel gets samples, min_spp first and then step_spp per pass,
        until its own standard error is <= rel_noise x its mean radiance + abs_noise (judged over its 3 x 3 neighbourhood),
        or it reaches the render's sample count (sample_count, else the camera's spp; at most 2^16).  Returns
        (mean, m2, spp, stats): each pixel's planes are the bits render_moments returns for a uniform render of spp[y, x]
        samples (sums with FLAG_SUM); spp is uint32."""
        cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
        h, w = int(cam["image_h"][0]), int(cam["image_w"][0])
        mean = np.empty((h, w, 3), dtype=np.float32)
        m2 = np.empty((h, w, 3), dtype=np.float32)
        spp = np.empty((h, w), dtype=np.uint32)
        opts = RenderOpts(seed, sample_offset, sample_count, VARIANT_MEGAKERNEL, flags)
        aopts = AdaptiveOpts(min_spp, step_spp, rel_noise, abs_noise)
        st = Stats()
        _check(lib().b200rt_render_adaptive(self._h, cam.ctypes.data, C.byref(opts), C.byref(aopts), mean.ctypes.data,
                                            m2.ctypes.data, spp.ctypes.data, C.byref(st)))
        return mean, m2, spp, st.as_dict()

    def bounds_violations(self) -> np.ndarray:
        """[stack, node index, primitive / material index, pixel] violations counted by a -DB200RT_DEBUG_BOUNDS build."""
        out = np.zeros(4, dtype=np.uint64)
        _check(lib().b200rt_debug_bounds(self._h, out.ctypes.data))
        return out

    def lane_accounting(self, cam: np.ndarray, seed: int = 0xB200, sample_offset: int = 0, sample_count: int = 0, flags: int = 0) -> np.ndarray:
        """Per-warp lane accounting of the default kernel's schedule (b200rt_debug_lane_accounting): 16 counters."""
        cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
        opts = RenderOpts(seed, sample_offset, sample_count, 0, flags)
        out = np.zeros(16, dtype=np.uint64)
        _check(lib().b200rt_debug_lane_accounting(self._h, cam.ctypes.data, C.byref(opts), out.ctypes.data))
        return out

    def render_device(self, cam: np.ndarray, out_ptr: int, stream: int = 0, seed: int = 0xB200, sample_offset: int = 0,
                      sample_count: int = 0, variant: int = VARIANT_MEGAKERNEL, flags: int = 0, want_stats: bool = True):
        """Renders into a DEVICE buffer (e.g. a torch tensor's data_ptr()) on `stream`."""
        cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
        opts = RenderOpts(seed, sample_offset, sample_count, variant, flags)
        st = Stats()
        _check(lib().b200rt_render_device(self._h, cam.ctypes.data, C.byref(opts), C.c_void_p(out_ptr),
                                          C.c_void_p(stream), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None


def render_scene(scene: HostScene, cam: np.ndarray, seed: int = 0xB200, sample_offset: int = 0, sample_count: int = 0,
                 variant: int = VARIANT_MEGAKERNEL, flags: int = 0, out: np.ndarray | None = None, devices=None):
    """The one-call drop-in for Camera::render(const Scene&): build + upload + render + read back.
    `devices`: list of CUDA ordinals -> b200rt_render_scene_multi (sample split across them inside the library)."""
    cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
    h, w = int(cam["image_h"][0]), int(cam["image_w"][0])
    if out is None:
        out = np.empty((h, w, 3), dtype=np.float32)
    desc = scene.desc()
    opts = RenderOpts(seed, sample_offset, sample_count, variant, flags)
    st, info = Stats(), SceneInfo()
    if devices is not None:
        devs = (C.c_int32 * len(devices))(*[int(d) for d in devices])
        _check(lib().b200rt_render_scene_multi(C.byref(desc), cam.ctypes.data, C.byref(opts), None, devs, len(devices),
                                               out.ctypes.data, C.byref(st), C.byref(info)))
    else:
        _check(lib().b200rt_render_scene(C.byref(desc), cam.ctypes.data, C.byref(opts), None, out.ctypes.data,
                                         C.byref(st), C.byref(info)))
    return out, st.as_dict(), info.as_dict()


def sample_variance(mean, m2, n: int) -> np.ndarray:
    """Per-pixel, per-channel sample variance s^2 = n/(n-1) * (m2 - mean^2) from render_moments' MEAN planes over n
    samples, in float64, clamped at 0 (FP32 rounding can push m2 - mean^2 slightly below 0); inf where n < 2.  The
    standard error of the pixel mean is sqrt(s^2 / n)."""
    mean = np.asarray(mean, dtype=np.float64)
    m2 = np.asarray(m2, dtype=np.float64)
    if n < 2:
        return np.full(np.broadcast(mean, m2).shape, np.inf)
    return np.maximum(n / (n - 1) * (m2 - mean * mean), 0.0)


def debug_philox(counters_keys: np.ndarray, device: int = 0) -> np.ndarray:
    """Philox4x32-10 as the kernels evaluate it, on the device: rows of (c0, c1, c2, c3, k0, k1) -> rows of 4 words."""
    ck = np.ascontiguousarray(counters_keys, dtype=np.uint32).reshape(-1, 6)
    out = np.empty((ck.shape[0], 4), dtype=np.uint32)
    _check(lib().b200rt_debug_philox(ck.ctypes.data, ck.shape[0], out.ctypes.data, device))
    return out


def debug_samplers(rnd_pairs: np.ndarray, device: int = 0):
    """The kernels' unit-sphere and unit-disk samplers for rows of two random words: (n x 3, n x 2) doubles."""
    rnd = np.ascontiguousarray(rnd_pairs, dtype=np.uint32).reshape(-1, 2)
    sph = np.empty((rnd.shape[0], 3), dtype=np.float64)
    disk = np.empty((rnd.shape[0], 2), dtype=np.float64)
    _check(lib().b200rt_debug_samplers(rnd.ctypes.data, rnd.shape[0], sph.ctypes.data, disk.ctypes.data, device))
    return sph, disk


def debug_camera_rays(cam: np.ndarray, pixels_xy: np.ndarray, rnd: np.ndarray, device: int = 0) -> np.ndarray:
    """The kernels' primary rays for the given (col, row) pixels and random words (b200rt_debug_camera_rays)."""
    cam = np.ascontiguousarray(cam, dtype=CAMERA_DTYPE).reshape(1)
    pixels_xy = np.ascontiguousarray(pixels_xy, dtype=np.uint32).reshape(-1, 2)
    rnd = np.ascontiguousarray(rnd, dtype=np.uint32).reshape(-1, 4)
    out = np.empty((pixels_xy.shape[0], 6), dtype=np.float64)
    _check(lib().b200rt_debug_camera_rays(cam.ctypes.data, pixels_xy.ctypes.data, rnd.ctypes.data, pixels_xy.shape[0],
                                          out.ctypes.data, device))
    return out


def tonemap(hdr: np.ndarray, clamp: bool = False) -> np.ndarray:
    hdr = np.ascontiguousarray(hdr, dtype=np.float32)
    n = hdr.size // 3
    out = np.empty(hdr.shape, dtype=np.int32)
    _check(lib().b200rt_tonemap(hdr.ctypes.data, n, out.ctypes.data, int(clamp)))
    return out
