"""GPU parity on the two multi-million-primitive configs (C4b raining_on_the_dance_floor:
2.2 M light quads + 25 k spheres; C5 millions_of_spheres_with_lights: 3.1 M spheres) and on the
host C++ layer's render call.  The scenes are built by the repo's own host code
(host/b200rt_scenes, pinned byte-for-byte against reference dumps in test_host_api_cpu.py); the
full comparison runs the compiled reference (oracle/_ref/ref_bridge) live because its fixtures
would be hundreds of MB; a stored sample of rays with their Scene::hit_by answers
(tests/golden/<scene>.rays.gz / .hits_brute.gz) checks the ray cast without it."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scenes_bin():
    from cpp_raytracer_b200 import build
    return build.build_host()


def _bridge(ref_bridge, args):
    res = subprocess.run([ref_bridge, *args], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    return [json.loads(l) for l in res.stdout.splitlines() if l.startswith("{")]


def tone(img):
    img = np.asarray(img, dtype=np.float64)
    lum = 0.2126 * img[..., 0] + 0.7152 * img[..., 1] + 0.0722 * img[..., 2]
    return np.sqrt(np.clip(img / (1.0 + lum[..., None]), 0, None))


@pytest.mark.parametrize("name,spp", [("raining", 64), ("millions_lights", 128)])
def test_big_scene_raycast_and_render_vs_reference(scenes_bin, ref_bridge, name, spp, tmp_path):
    if ref_bridge is None:
        pytest.skip("oracle/_ref/ref_bridge not built")
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import scene_io
    w, h = 160, 90
    scene_path = str(tmp_path / "s.scene")
    subprocess.run([scenes_bin, name, "dump", scene_path], check=True, capture_output=True)
    scene = scene_io.load_scene(scene_path)
    # ray set: camera rays (fixed jitter table) + rays the reference's own paths issue
    rec, rays_path, hits, hits_brute = (str(tmp_path / f) for f in ("rec.bin", "rays.bin", "hits.bin", "hits_brute.bin"))
    a_hdr, b_hdr = str(tmp_path / "a.hdr"), str(tmp_path / "b.hdr")
    small = str(tmp_path / "small.bin")
    cam_rays = scene_io.camera_rays(scene.camera, 150_000, seed=11)
    # one reference process: record secondary rays, then cast everything, then two independent renders
    scene_io.save_rays(small, cam_rays[:192])
    out = _bridge(ref_bridge, [name, "--w", str(w), "--h", str(h), "--spp", str(spp), "--render-seed", "77",
                               "record", "50000", "3", rec])
    rec_rays, _, _ = scene_io.load_rays(rec)
    rays = np.concatenate([cam_rays, rec_rays])
    scene_io.save_rays(rays_path, rays)
    out = _bridge(ref_bridge, [name, "--w", str(w), "--h", str(h), "--spp", str(spp), "--render-seed", "78",
                               "raycast", rays_path, hits, "raycast", small, hits_brute, "brute",
                               "render", a_hdr, "render", b_hdr])
    want_p, want_t = scene_io.load_hits(hits)
    bp, bt = scene_io.load_hits(hits_brute)
    with rt.DeviceSceneHandle(scene) as dev:
        info = dev.info()
        p, t = dev.raycast(rays)
        diff = np.nonzero((p != want_p) | (t != want_t))[0]
        ties = (t[diff] == want_t[diff]) & (p[diff] >= 0) & (want_p[diff] >= 0)
        print(f"{name}: {len(rays)} rays, hit frac {np.mean(want_p >= 0):.3f}, {len(diff)} differ from BVH::hit_by "
              f"({int(ties.sum())} exact ties); nodes {info['n_nodes']}, depth {info['tree_depth']}, "
              f"build {info['build_ms']:.0f} ms, device {info['device_bytes'] / 1e6:.0f} MB")
        assert np.all(ties), f"{name}: non-tie disagreement with the reference's BVH::hit_by"
        assert np.all(np.abs(t - want_t)[want_p >= 0] <= 1e-5 * np.abs(want_t[want_p >= 0]))
        assert np.array_equal(p[:192], bp) and np.array_equal(t[:192], bt)      # Scene::hit_by subset: exact
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp)
        G, st = dev.render(cam, seed=5)
    A, B = scene_io.load_hdr(a_hdr), scene_io.load_hdr(b_hdr)
    tA, tB, tG = tone(A), tone(B), tone(G)
    rm = lambda x, y: float(np.sqrt(np.mean((x - y) ** 2)))  # noqa: E731
    floor, got = rm(tA, tB), max(rm(tG, tA), rm(tG, tB))
    lum = lambda a: float((0.2126 * a[..., 0] + 0.7152 * a[..., 1] + 0.0722 * a[..., 2]).mean())  # noqa: E731
    lerr = abs(lum(tG) - 0.5 * (lum(tA) + lum(tB))) / (0.5 * (lum(tA) + lum(tB)))
    print(f"{name}: render RMSE {got:.5f} vs ref-vs-ref floor {floor:.5f} (ratio {got / floor:.3f}); mean luminance err {lerr:.3%}; "
          f"rays/path {st['rays'] / st['paths']:.3f}; {st['paths'] / st['kernel_ms'] / 1e3:.0f} Mpaths/s at {w}x{h}")
    assert got <= 1.25 * floor
    assert lerr <= 0.03 + 3 * abs(lum(tA) - lum(tB)) / lum(tA)


@pytest.mark.parametrize("name", ["raining", "millions_lights"])
def test_big_scene_raycast_matches_stored_scene_hit_by(scenes_bin, golden, name, tmp_path):
    """Camera rays and one bounce from each camera hit (tests/golden/make_big_golden.py) against Scene::hit_by
    as the oracle's C restatement answers it: primitive index and t bit-exact on every ray."""
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import scene_io
    scene_path = str(tmp_path / "s.scene")
    subprocess.run([scenes_bin, name, "dump", scene_path], check=True, capture_output=True)
    scene = scene_io.load_scene(scene_path)
    rays, tmin, tmax = golden.rays(name)
    want_p, want_t = golden.hits(name, brute=True)
    with rt.DeviceSceneHandle(scene) as dev:
        p, t = dev.raycast(rays, tmin, tmax)
    bad = np.nonzero((p != want_p) | (t != want_t))[0]
    assert len(bad) == 0, (f"{name}: {len(bad)} of {len(rays)} rays differ from Scene::hit_by; first: ray {bad[0]} "
                           f"got ({p[bad[0]]}, {t[bad[0]]!r}) want ({want_p[bad[0]]}, {want_t[bad[0]]!r})")


def test_host_cpp_render_call_writes_reference_format_ppm(scenes_bin, golden, tmp_path):
    """Camera::render(world).send_as_ppm(path) through the C++ mirror: a P3 file whose integers are
    exactly the tone-mapped pixels of the same render through the Python binding (same RNG key)."""
    import cpp_raytracer_b200 as rt
    ppm = str(tmp_path / "q.ppm")
    res = subprocess.run([scenes_bin, "quads", "--w", "48", "--h", "40", "--spp", "16", "render", ppm], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    tok = open(ppm).read().split()
    assert tok[0] == "P3" and tok[1:4] == ["48", "40", "255"]
    got = np.array(tok[4:], dtype=np.int32).reshape(40, 48, 3)
    scene = golden.scene("quads")
    with rt.DeviceSceneHandle(scene) as dev:
        img, _ = dev.render(rt.camera_with(scene.camera, image_w=48, image_h=40, spp=16), seed=0xB200)
    assert np.array_equal(got, rt.tonemap(img))


@pytest.mark.parametrize("name,w,h,spp", [("rtow_lights", 1920, 1080, 16), ("xmas", 1920, 1080, 8),
                                          ("cornell", 1024, 1024, 16), ("millions_lights", 3840, 2160, 4)])
def test_full_resolution_frame_converges_to_live_reference(scenes_bin, ref_bridge, name, w, h, spp, tmp_path):
    """BASELINE-size frames (C2 / C4 resolution, C3's 1024^2 at depth 1000, C5's 3840x2160 over 3.1 M spheres) against
    two live reference renders of the same size: the GPU-vs-reference RMSE sits on the reference-vs-reference noise
    floor."""
    if ref_bridge is None:
        pytest.skip("oracle/_ref/ref_bridge not built")
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import scene_io
    scene_path = str(tmp_path / "s.scene")
    subprocess.run([scenes_bin, name, "dump", scene_path], check=True, capture_output=True)
    scene = scene_io.load_scene(scene_path)
    a_hdr, b_hdr = str(tmp_path / "a.hdr"), str(tmp_path / "b.hdr")
    _bridge(ref_bridge, [name, "--w", str(w), "--h", str(h), "--spp", str(spp), "--render-seed", "31", "render", a_hdr, "render", b_hdr])
    with rt.DeviceSceneHandle(scene) as dev:
        G, st = dev.render(rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp), seed=77)
    tA, tB, tG = tone(scene_io.load_hdr(a_hdr)), tone(scene_io.load_hdr(b_hdr)), tone(G)
    rm = lambda x, y: float(np.sqrt(np.mean((x - y) ** 2)))  # noqa: E731
    floor, got = rm(tA, tB), max(rm(tG, tA), rm(tG, tB))
    blk = lambda a: a[: h // 8 * 8, : w // 8 * 8].reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3))  # noqa: E731
    floor_b, got_b = rm(blk(tA), blk(tB)), max(rm(blk(tG), blk(tA)), rm(blk(tG), blk(tB)))
    print(f"{name} {w}x{h}x{spp}: RMSE {got:.5f} vs floor {floor:.5f} ({got / floor:.3f}); 8x8 blocks {got_b:.5f} vs {floor_b:.5f} ({got_b / floor_b:.3f})")
    assert got <= 1.10 * floor and got_b <= 1.15 * floor_b
