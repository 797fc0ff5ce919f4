"""GPU tests of the path kernel's chunked tail: the last tiles of the grid are rendered by several blocks, each taking a
chunk of the tile's samples, and the last chunk to finish writes the pixels (kernels.cu block_work / pool_merge_chunk).

Every contribution is summed as 64-bit fixed point with integer additions, so how a tile's samples are divided among
blocks cannot change a bit of the frame.  B200RT_TAIL_TILES=0 gives whole tiles only; B200RT_TAIL_TILES=R,K forces R tail
tiles of K chunks.  Every frame here must be byte-identical to the whole-tile one."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

ALL = 1 << 30     # more tail tiles than any image here has: every tile is chunked

# (R, K) settings: all tiles in 1-sample chunks (8-sample ones under group_shift 3), ragged 7-sample chunks of 20 samples,
# one chunk per tile (the merge path with whole tiles), a few tail tiles, and the default plan.
FORCED = [f"{ALL},1000000", f"{ALL},3", f"{ALL},1", "5,4", None]


def with_tail(monkeypatch, setting, fn):
    if setting is None:
        monkeypatch.delenv("B200RT_TAIL_TILES", raising=False)
    else:
        monkeypatch.setenv("B200RT_TAIL_TILES", setting)
    try:
        return fn()
    finally:
        monkeypatch.delenv("B200RT_TAIL_TILES", raising=False)


@pytest.mark.parametrize("name", ["rtow_lights", "rtow_final", "cornell"])
@pytest.mark.parametrize("group_shift", ["0", "3"])
def test_tail_chunks_give_the_same_bits(golden, monkeypatch, name, group_shift):
    import cpp_raytracer_b200 as rt
    scene = golden.scene(name)
    monkeypatch.setenv("B200RT_GROUP_SHIFT", group_shift)
    with rt.DeviceSceneHandle(scene) as dev:
        # ragged edge tiles (203 x 117), and fewer tiles than the GPU holds blocks at once
        for (w, h, spp) in ((203, 117, 20), (61, 43, 9)):
            cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=25)
            want, st0 = with_tail(monkeypatch, "0", lambda: dev.render(cam, seed=7))
            for setting in FORCED:
                got, st = with_tail(monkeypatch, setting, lambda: dev.render(cam, seed=7))
                assert got.tobytes() == want.tobytes(), (name, group_shift, w, h, spp, setting)
                assert st["rays"] == st0["rays"] and st["paths"] == st0["paths"], setting


def test_tail_chunks_with_accumulate_and_a_sample_offset(golden, monkeypatch):
    import torch
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene("rtow_lights")
    cam = rt.camera_with(scene.camera, image_w=100, image_h=70, spp=13, max_depth=20)
    start = torch.rand((70, 100, 3), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    with rt.DeviceSceneHandle(scene) as dev:
        def run():
            out = start.clone()
            dev.render_device(cam, out.data_ptr(), seed=3, sample_offset=1000, flags=capi.FLAG_ACCUMULATE)
            torch.cuda.synchronize()
            return out.cpu().numpy()
        want = with_tail(monkeypatch, "0", run)
        for setting in FORCED:
            assert with_tail(monkeypatch, setting, run).tobytes() == want.tobytes(), setting


def test_tail_chunks_with_moments(golden, monkeypatch):
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_lights")
    cam = rt.camera_with(scene.camera, image_w=203, image_h=117, spp=20, max_depth=25)
    with rt.DeviceSceneHandle(scene) as dev:
        mean0, m20, _ = with_tail(monkeypatch, "0", lambda: dev.render_moments(cam, seed=5))
        for setting in FORCED:
            mean, m2, _ = with_tail(monkeypatch, setting, lambda: dev.render_moments(cam, seed=5))
            assert mean.tobytes() == mean0.tobytes() and m2.tobytes() == m20.tobytes(), setting


def test_tail_chunks_across_a_launch_split(golden, monkeypatch):
    """A tiny image over 2^16 samples with moments: three launches, each chunked on its own."""
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_lights")
    cam = rt.camera_with(scene.camera, image_w=9, image_h=5, spp=(2 << 16) + 37, max_depth=4)
    with rt.DeviceSceneHandle(scene) as dev:
        mean0, m20, st0 = with_tail(monkeypatch, "0", lambda: dev.render_moments(cam, seed=3))
        assert st0["kernel_launches"] == 3
        for setting in (f"{ALL},7", f"{ALL},1", None):
            mean, m2, st = with_tail(monkeypatch, setting, lambda: dev.render_moments(cam, seed=3))
            assert mean.tobytes() == mean0.tobytes() and m2.tobytes() == m20.tobytes(), setting
            assert st["kernel_launches"] == 3


def test_tail_chunks_keep_the_traversal_counters(golden, monkeypatch):
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    scene = golden.scene("cornell")
    cam = rt.camera_with(scene.camera, image_w=120, image_h=90, spp=11, max_depth=30)
    keys = ("rays", "node_visits", "prim_tests", "quad_tests")
    with rt.DeviceSceneHandle(scene) as dev:
        img0, st0 = with_tail(monkeypatch, "0", lambda: dev.render(cam, seed=2, flags=capi.FLAG_COUNTERS))
        for setting in FORCED:
            img, st = with_tail(monkeypatch, setting, lambda: dev.render(cam, seed=2, flags=capi.FLAG_COUNTERS))
            assert img.tobytes() == img0.tobytes(), setting
            assert [st[k] for k in keys] == [st0[k] for k in keys], setting


def test_tail_scratch_is_clean_between_renders(golden, monkeypatch):
    """Renders in a row on one handle with different chunkings, with and without the moments plane (whose partial sums are
    twice as large): each launch must leave the scratch zero for the next."""
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_final")
    cam = rt.camera_with(scene.camera, image_w=150, image_h=80, spp=17, max_depth=10)
    small = rt.camera_with(cam, image_w=40, image_h=30)
    with rt.DeviceSceneHandle(scene) as dev:
        want = with_tail(monkeypatch, "0", lambda: dev.render(cam, seed=4)[0])
        want_m = with_tail(monkeypatch, "0", lambda: dev.render_moments(cam, seed=4)[:2])
        want_small = with_tail(monkeypatch, "0", lambda: dev.render(small, seed=4)[0])
        for setting in (f"{ALL},3", f"{ALL},5", "3,2", f"{ALL},17", None):
            assert with_tail(monkeypatch, setting, lambda: dev.render(cam, seed=4)[0]).tobytes() == want.tobytes(), setting
            m = with_tail(monkeypatch, setting, lambda: dev.render_moments(cam, seed=4)[:2])
            assert m[0].tobytes() == want_m[0].tobytes() and m[1].tobytes() == want_m[1].tobytes(), setting
            assert with_tail(monkeypatch, setting, lambda: dev.render(small, seed=4)[0]).tobytes() == want_small.tobytes(), setting


def test_tail_chunks_on_a_multi_device_handle(golden, monkeypatch):
    import cpp_raytracer_b200 as rt
    scene = golden.scene("rtow_lights")
    cam = rt.camera_with(scene.camera, image_w=64, image_h=36, spp=16)
    with rt.DeviceSceneHandle(scene, devices=[0, 0]) as dm:
        img0, st0 = with_tail(monkeypatch, "0", lambda: dm.render(cam, seed=9))
        mean0, m20, _ = with_tail(monkeypatch, "0", lambda: dm.render_moments(cam, seed=9))
        assert st0["n_devices"] == 2
        for setting in FORCED:
            assert with_tail(monkeypatch, setting, lambda: dm.render(cam, seed=9)[0]).tobytes() == img0.tobytes(), setting
            mean, m2, _ = with_tail(monkeypatch, setting, lambda: dm.render_moments(cam, seed=9))
            assert mean.tobytes() == mean0.tobytes() and m2.tobytes() == m20.tobytes(), setting


BOUNDS_CHILD = r'''
import json, os, sys, hashlib
sys.path.insert(0, os.environ["B200RT_ROOT"])
import cpp_raytracer_b200 as rt
from cpp_raytracer_b200 import scene_io
g = os.path.join(os.environ["B200RT_ROOT"], "tests", "golden")
out = {}
for name in ("rtow_lights", "cornell"):
    scene = scene_io.load_scene(os.path.join(g, name + ".scene.gz"))
    cam = rt.camera_with(scene.camera, image_w=61, image_h=43, spp=9, max_depth=12)
    with rt.DeviceSceneHandle(scene) as dev:
        res = {}
        for setting in ("0", "1073741824,9", "1073741824,2", "3,3"):
            os.environ["B200RT_TAIL_TILES"] = setting
            img, st = dev.render(cam, seed=3)
            mean, m2, _ = dev.render_moments(cam, seed=3)
            res[setting] = [hashlib.sha256(x.tobytes()).hexdigest() for x in (img, mean, m2)]
        try:
            viol = [int(x) for x in dev.bounds_violations()]
        except rt.B200rtError:
            viol = None
    out[name] = {"viol": viol, "frames": res}
print(json.dumps(out))
'''


def test_tail_chunks_under_the_bounds_checked_build():
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
