#!/usr/bin/env python
"""Generates the committed fixtures of the two multi-million-primitive scenes (raining: 2.2 M quads +
25 k spheres; millions_lights: 3.1 M spheres).  Their scene files are hundreds of MB, so only a digest
and a small ray sample are kept:

    python tests/golden/make_big_golden.py        # needs the in-tree build (libb200rt.so, host/b200rt_scenes)

    big_scenes.json         byte length + SHA-256 of each scene as host/b200rt_scenes dumps it
    <scene>.rays.gz         camera rays (fixed jitter table) + one bounce from each camera hit in a
                            seeded random direction
    <scene>.hits_brute.gz   (prim, t) of those rays through Scene::hit_by semantics, from the oracle's
                            C restatement (oracle/pt_oracle.c, pinned bit for bit against the reference's
                            Scene::hit_by on the small scenes by tests/test_oracle_cpu.py)
"""
import gzip
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from cpp_raytracer_b200 import build, scene_io  # noqa: E402
import pt_oracle  # noqa: E402

BIG_SCENES = ["raining", "millions_lights"]
N_CAMERA_RAYS = 768


def bounce_rays(rays, prim, t, rng):
    """One ray from every hit point, in a uniformly random direction."""
    hit = prim >= 0
    o = rays[hit, :3] + t[hit, None] * rays[hit, 3:]
    d = rng.normal(size=o.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d], axis=1)


def main():
    scenes_bin = build.build_host()
    digests = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name in BIG_SCENES:
            path = os.path.join(tmp, f"{name}.scene")
            subprocess.run([scenes_bin, name, "dump", path], check=True, capture_output=True)
            with open(path, "rb") as f:
                data = f.read()
            digests[name] = {"bytes": len(data), "sha256": hashlib.sha256(data).hexdigest()}
            scene = scene_io.load_scene(path)
            cam_rays = scene_io.camera_rays(scene.camera, N_CAMERA_RAYS, seed=11)
            p, t = pt_oracle.raycast_brute(scene, cam_rays)
            rays = np.concatenate([cam_rays, bounce_rays(cam_rays, p, t, np.random.default_rng(12))])
            p, t = pt_oracle.raycast_brute(scene, rays)
            scene_io.save_rays(os.path.join(HERE, f"{name}.rays.gz"), rays)
            with gzip.open(os.path.join(HERE, f"{name}.hits_brute.gz"), "wb") as f:
                f.write(p.astype("<i4").tobytes() + t.astype("<f8").tobytes())
            print(f"{name}: {len(data)} bytes, {len(rays)} rays, hit frac {np.mean(p >= 0):.3f}")
    with open(os.path.join(HERE, "big_scenes.json"), "w") as f:
        json.dump(digests, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
