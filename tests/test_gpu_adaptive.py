"""GPU tests of adaptive sampling (b200rt_render_adaptive, DeviceSceneHandle.render_adaptive, the host layer's
Camera::render_adaptive).

Each pixel's sums are kept as int64 fixed point across passes, so a pixel that ends with n samples has the same integer
sums as a uniform render of n samples and must come back with the same bits in both planes.  The convergence rule is
exact (double, no FMA), so the per-pixel counts are replayed here pass by pass from uniform renders."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

ALL = 1 << 30     # more tail tiles than any image here has: every tile of every pass is chunked


def with_tail(monkeypatch, setting, fn):
    if setting is None:
        monkeypatch.delenv("B200RT_TAIL_TILES", raising=False)
    else:
        monkeypatch.setenv("B200RT_TAIL_TILES", setting)
    try:
        return fn()
    finally:
        monkeypatch.delenv("B200RT_TAIL_TILES", raising=False)


def pass_counts(min_spp, step_spp, max_spp):
    """The sample count of the active pixels after each pass."""
    n = [min(min_spp, max_spp)]
    while n[-1] < max_spp:
        n.append(n[-1] + min(step_spp, max_spp - n[-1]))
    return n


def converged(mean, m2, n, rel, abs_):
    """The rule of b200rt_render_adaptive on MEAN planes over n samples, in float64 in the library's operation order."""
    mean = np.asarray(mean, np.float32).astype(np.float64)
    m2 = np.asarray(m2, np.float32).astype(np.float64)
    d = m2 - mean * mean
    var = np.where(d <= m2 * 2.0 ** -20 + 2.0 ** -24, 0.0, (n / (n - 1)) * d)
    err = np.sqrt((var[..., 0] + var[..., 1] + var[..., 2]) / (3.0 * n))
    level = (mean[..., 0] + mean[..., 1] + mean[..., 2]) / 3.0
    return err <= rel * level + abs_


def dilate(mask):
    h, w = mask.shape
    p = np.zeros((h + 2, w + 2), bool)
    p[1:-1, 1:-1] = mask
    out = np.zeros_like(mask)
    for dy in range(3):
        for dx in range(3):
            out |= p[dy:dy + h, dx:dx + w]
    return out


def replay(uniform, min_spp, step_spp, max_spp, rel, abs_):
    """Per-pixel counts of an adaptive render, from uniform MEAN renders {n: (mean, m2)} at every pass count."""
    counts = pass_counts(min_spp, step_spp, max_spp)
    h, w = uniform[counts[0]][0].shape[:2]
    active = np.ones((h, w), bool)
    spp = np.full((h, w), counts[0], np.uint32)
    for n, n_next in zip(counts, counts[1:]):
        mean, m2 = uniform[n]
        active &= dilate(active & ~converged(mean, m2, n, rel, abs_))   # stopped pixels were converged: they add nothing
        if not active.any():
            break
        spp[active] = n_next
    return spp


def uniform_renders(dev, cam, counts, seed, offset, flags=0):
    return {n: dev.render_moments(cam, seed=seed, sample_offset=offset, sample_count=n, flags=flags)[:2] for n in counts}


def target_for(uniform, counts):
    """A relative target that the median pixel meets about halfway through, so the counts spread over the passes."""
    n = counts[len(counts) // 2]
    mean, m2 = uniform[n]
    lvl = mean.astype(np.float64).mean(axis=-1)
    ok = lvl > 0
    lo, hi = 0.0, 10.0
    for _ in range(60):   # bisect on the share of converged pixels
        mid = 0.5 * (lo + hi)
        share = converged(mean, m2, n, mid, 0.0)[ok].mean() if ok.any() else 1.0
        lo, hi = (mid, hi) if share < 0.5 else (lo, mid)
    return hi


def check_against_uniform(got, spp, uniform_at):
    mean, m2 = got
    for c in np.unique(spp):
        sel = spp == c
        um, u2 = uniform_at[int(c)]
        assert mean[sel].tobytes() == um[sel].tobytes(), int(c)
        assert m2[sel].tobytes() == u2[sel].tobytes(), int(c)


# ---- exactness and the decision replay ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rtow_lights", "cornell", "xmas", "quads"])
@pytest.mark.parametrize("group_shift", ["0", "3"])
def test_adaptive_pixels_are_uniform_renders_and_the_counts_replay(golden, monkeypatch, name, group_shift):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene(name)
    monkeypatch.setenv("B200RT_GROUP_SHIFT", group_shift)
    min_spp, step, max_spp, seed, offset = 6, 12, 42, 17, 1000     # ragged against groups of 8 samples
    counts = pass_counts(min_spp, step, max_spp)
    with rt.DeviceSceneHandle(scene) as dev:
        for (w, h) in ((203, 117), (61, 43)):
            cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=max_spp, max_depth=25)
            uni = uniform_renders(dev, cam, counts, seed, offset)
            rel = target_for(uni, counts)
            mean, m2, spp, st = dev.render_adaptive(cam, rel, min_spp=min_spp, step_spp=step, seed=seed, sample_offset=offset)
            assert spp.dtype == np.uint32 and spp.shape == (h, w)
            assert np.array_equal(spp, replay(uni, min_spp, step, max_spp, rel, 0.0)), (name, w, h)
            assert len(np.unique(spp)) >= 2, np.unique(spp)
            check_against_uniform((mean, m2), spp, uni)
            assert st["paths"] == int(spp.sum(dtype=np.uint64))
            # sums: the same pixels, as SUM planes
            s, s2, spp_s, _ = dev.render_adaptive(cam, rel, min_spp=min_spp, step_spp=step, seed=seed, sample_offset=offset,
                                                  flags=capi.FLAG_SUM)
            assert np.array_equal(spp_s, spp)
            check_against_uniform((s, s2), spp, uniform_renders(dev, cam, np.unique(spp).tolist(), seed, offset, capi.FLAG_SUM))


@pytest.mark.parametrize("group_shift", ["0", "3"])
def test_adaptive_renders_are_the_same_under_every_tail_plan(golden, monkeypatch, group_shift):
    """Late passes have few tiles, so the chunked tail carries them; how a pass's tiles are split into sample chunks
    cannot change a bit."""
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_lights")
    monkeypatch.setenv("B200RT_GROUP_SHIFT", group_shift)
    with rt.DeviceSceneHandle(scene) as dev:
        for (w, h) in ((203, 117), (61, 43)):
            cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=40, max_depth=25)
            want = with_tail(monkeypatch, "0", lambda: dev.render_adaptive(cam, 0.3, min_spp=8, step_spp=5, seed=3, sample_offset=77))
            assert len(np.unique(want[2])) >= 2
            for setting in (f"{ALL},1000000", f"{ALL},3", f"{ALL},1", "5,4", None):
                got = with_tail(monkeypatch, setting, lambda: dev.render_adaptive(cam, 0.3, min_spp=8, step_spp=5, seed=3, sample_offset=77))
                for a, b in zip(got[:3], want[:3]):
                    assert a.tobytes() == b.tobytes(), (w, h, setting)
                assert got[3]["rays"] == want[3]["rays"] and got[3]["paths"] == want[3]["paths"], setting


# ---- limits ------------------------------------------------------------------------------------------------------
def test_limits_zero_target_huge_target_and_a_single_pass(golden):
    import cpp_raytracer_b200 as rt
    scene = golden.scene("cornell")
    with rt.DeviceSceneHandle(scene) as dev:
        # a zero target still stops a pixel whose whole 3 x 3 neighbourhood has exactly zero variance: on this view the light
        # seen directly, the black border outside the box, and dark corners whose first samples all came back black
        cam = rt.camera_with(scene.camera, image_w=96, image_h=80, spp=24, max_depth=30)
        full_mean, full_m2, full_st = dev.render_moments(cam, seed=5)
        mean, m2, spp, st = dev.render_adaptive(cam, 0.0, 0.0, min_spp=8, step_spp=8, seed=5)
        uni = uniform_renders(dev, cam, pass_counts(8, 8, 24), 5, 0)
        assert np.array_equal(spp, replay(uni, 8, 8, 24, 0.0, 0.0))
        assert (spp == 8).any() and (spp == 24).any()
        check_against_uniform((mean, m2), spp, uni)
        assert st["paths"] == int(spp.sum(dtype=np.uint64))
        # a target every pixel meets: the uniform min_spp render
        mean, m2, spp, st = dev.render_adaptive(cam, 1e30, min_spp=8, step_spp=8, seed=5)
        m8, m28, st8 = dev.render_moments(cam, seed=5, sample_count=8)
        assert (spp == 8).all() and mean.tobytes() == m8.tobytes() and m2.tobytes() == m28.tobytes()
        assert st["rays"] == st8["rays"] and st["paths"] == st8["paths"]
        # min_spp == the maximum: one pass (init, path, judge, finish kernels), the uniform render at the maximum
        mean, m2, spp, st = dev.render_adaptive(cam, 0.0, min_spp=24, step_spp=8, seed=5)
        assert (spp == 24).all() and mean.tobytes() == full_mean.tobytes() and m2.tobytes() == full_m2.tobytes()
        assert st["kernel_launches"] == 4 and st["rays"] == full_st["rays"] and st["paths"] == full_st["paths"]
        # a maximum below min_spp: every pixel gets the maximum in the first pass
        mean, m2, spp, _ = dev.render_adaptive(cam, 0.0, min_spp=32, step_spp=8, seed=5)
        assert (spp == 24).all() and mean.tobytes() == full_mean.tobytes()


def test_zero_rays_with_an_exact_count_of_zero(golden):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene("cornell")
    with rt.DeviceSceneHandle(scene) as dev:
        cam = rt.camera_with(scene.camera, image_w=33, image_h=21, spp=24)
        mean, m2, spp, st = dev.render_adaptive(cam, 0.1, sample_count=0, flags=capi.FLAG_EXACT_COUNT)
        assert not mean.any() and not m2.any() and not spp.any() and st["paths"] == 0 and st["rays"] == 0


def test_background_pixels_stop_at_min_spp(golden):
    """rtow_final's sky has exactly zero variance after any number of samples: a sky pixel whose 3 x 3 neighbourhood is
    all sky stops after the first pass, whatever the target."""
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_final")
    with rt.DeviceSceneHandle(scene) as dev:
        cam = rt.camera_with(scene.camera, image_w=160, image_h=90, spp=48, max_depth=20)
        m, q, _ = dev.render_moments(cam, seed=2, sample_count=8)
        flat_hood = ~dilate(~converged(m, q, 8, 0.0, 0.0))   # the whole neighbourhood has zero variance at 8 samples
        assert flat_hood.sum() > 100
        mean, m2, spp, _ = dev.render_adaptive(cam, 0.0, min_spp=8, step_spp=8, seed=2)
        assert (spp[flat_hood] == 8).all()
        assert (spp[~flat_hood] == 48).all()          # a zero target keeps every noisy neighbourhood to the maximum
        assert mean[flat_hood].tobytes() == m[flat_hood].tobytes() and m2[flat_hood].tobytes() == q[flat_hood].tobytes()


# ---- stats and errors --------------------------------------------------------------------------------------------
def test_rejected_options_and_handles(golden):
    import ctypes
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene("rtow_lights")
    cam = rt.camera_with(scene.camera, image_w=16, image_h=8, spp=16)
    with rt.DeviceSceneHandle(scene) as dev:
        for flags in (capi.FLAG_THREAD_PIXELS, capi.FLAG_COUNTERS):
            with pytest.raises(rt.B200rtError) as e:
                dev.render_adaptive(cam, 0.1, flags=flags)
            assert e.value.code == capi.EINVAL
        bad = [dict(min_spp=1), dict(min_spp=0), dict(step_spp=0), dict(sample_count=(1 << 16) + 1),
               dict(rel_noise=-0.1), dict(rel_noise=float("nan")), dict(rel_noise=float("inf")),
               dict(abs_noise=-1e-9), dict(abs_noise=float("nan")), dict(abs_noise=float("inf"))]
        for kw in bad:
            args = dict(rel_noise=0.1)
            args.update(kw)
            with pytest.raises(rt.B200rtError) as e:
                dev.render_adaptive(cam, **args)
            assert e.value.code == capi.EINVAL, kw
        # the wavefront variant, through the C entry (the Python method always asks for the default kernel)
        c = np.ascontiguousarray(cam, dtype=capi.CAMERA_DTYPE).reshape(1)
        out = np.zeros((8, 16, 3), np.float32)
        opts = capi.RenderOpts(1, 0, 0, capi.VARIANT_WAVEFRONT, 0)
        aopts = capi.AdaptiveOpts(16, 16, 0.1, 0.0)
        assert capi.lib().b200rt_render_adaptive(dev._h, c.ctypes.data, ctypes.byref(opts), ctypes.byref(aopts), out.ctypes.data,
                                                 None, None, None) == capi.EINVAL
        opts = capi.RenderOpts(1, 0, 0, capi.VARIANT_MEGAKERNEL, 0)
        assert capi.lib().b200rt_render_adaptive(dev._h, c.ctypes.data, ctypes.byref(opts), None, out.ctypes.data,
                                                 None, None, None) == capi.EINVAL
        # both optional planes may be left out
        assert capi.lib().b200rt_render_adaptive(dev._h, c.ctypes.data, ctypes.byref(opts), ctypes.byref(aopts), out.ctypes.data,
                                                 None, None, None) == capi.OK
        assert np.array_equal(out, dev.render_adaptive(cam, 0.1, seed=1)[0])
    with rt.DeviceSceneHandle(scene, devices=[0, 0]) as dm:
        with pytest.raises(rt.B200rtError) as e:
            dm.render_adaptive(cam, 0.1)
        assert e.value.code == capi.EINVAL


# ---- bounds-checked build ----------------------------------------------------------------------------------------
BOUNDS_CHILD = r'''
import json, os, sys, hashlib
sys.path.insert(0, os.environ["B200RT_ROOT"])
import cpp_raytracer_b200 as rt
from cpp_raytracer_b200 import scene_io
g = os.path.join(os.environ["B200RT_ROOT"], "tests", "golden")
out = {}
for name in ("rtow_lights", "cornell"):
    scene = scene_io.load_scene(os.path.join(g, name + ".scene.gz"))
    cam = rt.camera_with(scene.camera, image_w=61, image_h=43, spp=30, max_depth=12)
    with rt.DeviceSceneHandle(scene) as dev:
        res = {}
        for setting in ("0", "1073741824,9", "1073741824,2", "3,3"):
            os.environ["B200RT_TAIL_TILES"] = setting
            mean, m2, spp, st = dev.render_adaptive(cam, 0.2, min_spp=6, step_spp=4, seed=3)
            res[setting] = [hashlib.sha256(x.tobytes()).hexdigest() for x in (mean, m2, spp)] + [len(set(spp.ravel().tolist()))]
        try:
            viol = [int(x) for x in dev.bounds_violations()]
        except rt.B200rtError:
            viol = None
    out[name] = {"viol": viol, "frames": res}
print(json.dumps(out))
'''


def test_adaptive_under_the_bounds_checked_build():
    from cpp_raytracer_b200 import build

    def run(lib):
        env = dict(os.environ, B200RT_ROOT=ROOT, B200RT_LIB=lib)
        r = subprocess.run([sys.executable, "-c", BOUNDS_CHILD], capture_output=True, text=True, env=env)
        assert r.returncode == 0, r.stderr[-3000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    dbg = run(build.build_debug())
    prod = run(os.path.join(ROOT, "cpp_raytracer_b200", "libb200rt.so"))
    for name in dbg:
        assert dbg[name]["viol"] == [0, 0, 0, 0], (name, dbg[name]["viol"])
        assert prod[name]["viol"] is None
        frames = dbg[name]["frames"]
        for setting in frames:
            assert frames[setting] == frames["0"] == prod[name]["frames"][setting], (name, setting)
            assert frames[setting][3] >= 2        # the passes did stop pixels at different counts


# ---- host layer --------------------------------------------------------------------------------------------------
PROGRAM = r'''
#include <cstdio>
#include "util/rand_util.h"
#include "base/scene.h"
#include "base/material.h"
#include "base/camera.h"
#include "acceleration/bvh.h"
#include "shapes/shapes.h"

int main() {
    SeedSeqGenerator::get_instance().set_seed(7);
    Scene world;
    world.add(std::make_shared<Sphere>(Point3D(0, 0, 0), 1.0, std::make_shared<Dielectric>(1.5)));
    world.add(std::make_shared<Sphere>(Point3D(-1.5, -0.5, 0.5), 0.5, std::make_shared<Lambertian>(RGB::from_mag(0.5, 0.4, 0.3))));
    world.add(std::make_shared<Parallelogram>(Point3D(-2, -2, -3), Vec3D(4, 0, 0), Vec3D(0, 4, 0),
                                              std::make_shared<Metal>(RGB::from_mag(0.7, 0.6, 0.5), 0.1)));
    world.add(std::make_shared<Box>(Point3D(1.2, -1, 0), Point3D(1.8, -0.4, 0.6), std::make_shared<DiffuseLight>(RGB::from_mag(1), 4)));
    Camera cam;
    cam.set_image_dimensions(64, 48).set_vertical_fov(30).set_camera_center(Point3D{0, 0, 10})
       .set_camera_lookat(Point3D{0, 0, 0}).set_samples_per_pixel(48).set_max_depth(8).set_background(RGB::from_mag(0.7, 0.8, 1));
    std::vector<int32_t> devs{0};
    BVH bvh(world, 32, 12, devs);
    const auto [img, spp] = cam.render_adaptive(bvh, 0.05, 8, 8);
    const uint64_t paths = cam.stats().paths;

    const B200rtCamera c = cam.to_abi();
    B200rtRenderOpts o{};
    o.seed = 0xB200;
    B200rtAdaptiveOpts a{8, 8, 0.05, 0.0};
    std::vector<float> hdr(64 * 48 * 3);
    std::vector<uint32_t> spp_c(64 * 48);
    const int rc = b200rt_render_adaptive(bvh.handle(), &c, &o, &a, hdr.data(), nullptr, spp_c.data(), nullptr);
    const Image want = Camera::to_image(hdr, 64, 48);
    bool same = rc == B200RT_OK && spp == spp_c;
    for (size_t r = 0; r < 48; ++r)
        for (size_t col = 0; col < 64; ++col)
            if (img[r][col].r != want[r][col].r || img[r][col].g != want[r][col].g || img[r][col].b != want[r][col].b) same = false;
    uint64_t sum = 0;
    uint32_t lo = 0xFFFFFFFFu, hi = 0;
    for (uint32_t n : spp) { sum += n; lo = std::min(lo, n); hi = std::max(hi, n); }
    std::printf("{\"same\": %d, \"paths\": %llu, \"sum\": %llu, \"lo\": %u, \"hi\": %u}\n", (int)same,
                (unsigned long long)paths, (unsigned long long)sum, lo, hi);
    return 0;
}
'''


def compile_program(tmp_path):
    src = tmp_path / "adaptive.cpp"
    src.write_text(PROGRAM)
    exe = str(tmp_path / "adaptive")
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    inc = os.path.join(ROOT, "cpp_raytracer_b200", "host", "include")
    lib = os.path.join(ROOT, "cpp_raytracer_b200")
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{inc}", "-o", exe, str(src), f"-L{lib}", "-lb200rt", f"-Wl,-rpath,{lib}"],
                   check=True, env=env)
    return exe


def test_host_layer_render_adaptive(tmp_path):
    exe = compile_program(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    print(res)
    assert res["same"] == 1
    assert res["paths"] == res["sum"]
    assert res["lo"] == 8 and res["hi"] == 48     # the sky stops after the first pass; the noisiest pixels take all 48
