"""Scene-spanning primitives (bvh_builder.h spanning_key): a primitive whose box has at least half the surface area of the
scene's box is left out of the tree and tested by every ray before it (traverse.cuh trav_hoisted).  Which primitives
qualify is checked on the CPU; on the GPU, hoisting must not change a single bit of any hit, frame or ray count."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, RENDER_SCENES, SMALL_SCENES

# scene -> the array holding its ground, the one primitive expected to be hoisted
GROUNDS = {"rtow_final": "spheres", "rtow_lights": "spheres", "xmas": "quads"}


def _shrunk(scene, kind, index):
    """The scene with primitive `index` of `kind` shrunk to a tenth of its size about its centre (or corner)."""
    from cpp_raytracer_b200 import capi
    arrays = {"spheres": scene.spheres.copy(), "quads": scene.quads.copy()}
    if kind == "spheres":
        arrays[kind]["r"][index] *= 0.1
    else:
        arrays[kind]["s1"][index] *= 0.1
        arrays[kind]["s2"][index] *= 0.1
    return capi.HostScene(scene.materials, arrays["spheres"], arrays["quads"], scene.camera)


def _ground_index(scene, kind):
    """The ground: the sphere of largest radius, or the quad of largest |s1 x s2|."""
    if kind == "spheres":
        return int(np.argmax(scene.spheres["r"]))
    return int(np.argmax(np.linalg.norm(np.cross(scene.quads["s1"], scene.quads["s2"]), axis=1)))


@pytest.mark.parametrize("name", SMALL_SCENES)
def test_selection_hoists_exactly_the_ground(golden, name, monkeypatch):
    """The rule picks the ground of rtow_final, rtow_lights and xmas and nothing in cornell, cornell_empty, quads or
    pathological; validate_bvh4 checks that the tree covers exactly the primitives that were not hoisted."""
    import cpp_raytracer_b200 as rt
    scene = golden.scene(name)
    info = rt.selftest_bvh(scene)
    if name not in GROUNDS:
        assert info["n_hoisted"] == 0, name
        return
    assert info["n_hoisted"] == 1, name
    kind = GROUNDS[name]
    ground = _ground_index(scene, kind)
    # the one hoisted primitive is the ground: with the ground shrunk, nothing in the scene spans it any more
    assert rt.selftest_bvh(_shrunk(scene, kind, ground))["n_hoisted"] == 0, name
    monkeypatch.setenv("B200RT_HOISTED", "0")
    assert rt.selftest_bvh(scene)["n_hoisted"] == 0


@pytest.mark.parametrize("name,want", [("millions_lights", 1), ("raining", 0)])
def test_selection_on_the_generated_scenes(name, want, tmp_path):
    """C5's ground sphere (r = 1e6) is hoisted; nothing in raining is."""
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import build, scene_io
    path = str(tmp_path / f"{name}.scene")
    subprocess.run([build.build_host(), name, "dump", path], check=True, capture_output=True)
    scene = scene_io.load_scene(path)
    info = rt.selftest_bvh(scene)
    assert info["n_hoisted"] == want
    if want:
        ground = _ground_index(scene, "spheres")
        assert scene.spheres["r"][ground] == 1e6
        assert rt.selftest_bvh(_shrunk(scene, "spheres", ground))["n_hoisted"] == 0


def test_selection_keeps_one_primitive_in_the_tree_and_takes_the_largest_first():
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    cam = np.zeros(1, capi.CAMERA_DTYPE)
    mats = np.zeros(1, capi.MATERIAL_DTYPE)
    # six coincident spheres: every one spans the scene, four are hoisted and two stay in the tree
    sph = np.zeros(6, capi.SPHERE_DTYPE)
    sph["r"] = [9.0, 9.2, 9.4, 9.6, 9.8, 10.0]
    sph["prim"] = np.arange(6)
    assert rt.selftest_bvh(capi.HostScene(mats, sph, np.zeros(0, capi.QUAD_DTYPE), cam))["n_hoisted"] == 4
    # two: one is hoisted, one stays
    assert rt.selftest_bvh(capi.HostScene(mats, sph[:2], np.zeros(0, capi.QUAD_DTYPE), cam))["n_hoisted"] == 1
    # one: the tree keeps it
    assert rt.selftest_bvh(capi.HostScene(mats, sph[:1], np.zeros(0, capi.QUAD_DTYPE), cam))["n_hoisted"] == 0


def _builders():
    from cpp_raytracer_b200 import capi
    return {"host_sah": capi.BUILDER_HOST_SAH, "gpu_lbvh": capi.BUILDER_GPU_LBVH}


def _with_hoisting(on, monkeypatch):
    if on:
        monkeypatch.delenv("B200RT_HOISTED", raising=False)
    else:
        monkeypatch.setenv("B200RT_HOISTED", "0")


@pytest.mark.gpu
@pytest.mark.parametrize("builder", ["host_sah", "gpu_lbvh"])
@pytest.mark.parametrize("name", RENDER_SCENES)
def test_frame_is_the_same_bits_with_and_without_hoisting(golden, name, builder, monkeypatch):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene(name)
    cam = rt.camera_with(scene.camera, image_w=96, image_h=54, spp=16, max_depth=30)
    out = {}
    for on in (True, False):
        _with_hoisting(on, monkeypatch)
        with rt.DeviceSceneHandle(scene, builder=_builders()[builder]) as dev:
            hoisted = dev.info()["n_hoisted"]
            img, st = dev.render(cam, seed=29)
            img_c, st_c = dev.render(cam, seed=29, flags=capi.FLAG_COUNTERS)
            wf, st_wf = dev.render(cam, seed=29, variant=capi.VARIANT_WAVEFRONT)
        out[on] = (hoisted, img, st, img_c, st_c, wf, st_wf)
    assert out[True][0] == (1 if name in GROUNDS else 0) and out[False][0] == 0
    for k in (1, 3):
        assert np.array_equal(out[True][k], out[False][k]), (name, builder, k)
    for k in (2, 4, 6):
        assert out[True][k]["rays"] == out[False][k]["rays"], (name, builder, k)
    # the wavefront variant adds into the frame with atomics, so only the order of its FP32 additions may differ
    tol = 1e-4 * max(1.0, float(np.abs(out[False][5]).max()))
    assert np.allclose(out[True][5], out[False][5], rtol=2e-4, atol=tol), (name, builder)


@pytest.mark.gpu
@pytest.mark.parametrize("builder", ["host_sah", "gpu_lbvh"])
@pytest.mark.parametrize("name", SMALL_SCENES)
def test_closest_hits_match_the_reference_with_hoisting(golden, name, builder, monkeypatch):
    """The fixture rays, adversarial and far-field ground rays included, against the reference's Scene::hit_by."""
    import cpp_raytracer_b200 as rt
    monkeypatch.delenv("B200RT_HOISTED", raising=False)
    scene = golden.scene(name)
    rays, tmin, tmax = golden.rays(name)
    want_p, want_t = golden.hits(name, brute=True)
    with rt.DeviceSceneHandle(scene, builder=_builders()[builder]) as dev:
        assert dev.info()["n_hoisted"] == (1 if name in GROUNDS else 0)
        p, t = dev.raycast(rays, tmin, tmax)
    assert np.array_equal(p, want_p) and np.array_equal(t, want_t), (name, builder)


CHILD = r'''
import hashlib, json, os, sys
sys.path.insert(0, os.environ["B200RT_ROOT"])
import cpp_raytracer_b200 as rt
from cpp_raytracer_b200 import capi, scene_io
g = os.path.join(os.environ["B200RT_ROOT"], "tests", "golden")
out = {}
for name in os.environ["SCENES"].split(","):
    scene = scene_io.load_scene(os.path.join(g, name + ".scene.gz"))
    for builder in (capi.BUILDER_HOST_SAH, capi.BUILDER_GPU_LBVH):
        with rt.DeviceSceneHandle(scene, builder=builder) as dev:
            cam = rt.camera_with(scene.camera, image_w=64, image_h=48, spp=8, max_depth=12)
            img, st = dev.render(cam, seed=3)
            viol = [int(x) for x in dev.bounds_violations()]
            out[f"{name}/{builder}"] = {"viol": viol, "img": hashlib.sha256(img.tobytes()).hexdigest(), "rays": st["rays"],
                                        "n_hoisted": dev.info()["n_hoisted"]}
print(json.dumps(out))
'''


@pytest.mark.gpu
def test_bounds_checked_build_with_hoisting_sees_no_violation_and_the_same_frames():
    from cpp_raytracer_b200 import build
    lib = build.build_debug()
    got = {}
    for on in (True, False):
        env = dict(os.environ, B200RT_ROOT=ROOT, SCENES=",".join(RENDER_SCENES), B200RT_LIB=lib)
        if on:
            env.pop("B200RT_HOISTED", None)
        else:
            env["B200RT_HOISTED"] = "0"
        res = subprocess.run([sys.executable, "-c", CHILD], capture_output=True, text=True, env=env)
        assert res.returncode == 0, res.stderr[-3000:]
        got[on] = json.loads(res.stdout.strip().splitlines()[-1])
    for key, r in got[True].items():
        assert r["viol"] == [0, 0, 0, 0], (key, r["viol"])
        assert r["img"] == got[False][key]["img"] and r["rays"] == got[False][key]["rays"], key
        assert r["n_hoisted"] == (1 if key.split("/")[0] in GROUNDS else 0), key
