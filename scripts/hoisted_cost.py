#!/usr/bin/env python
"""Gain of testing the scene-spanning primitives before the tree (bvh_builder.h spanning_key, traverse.cuh trav_hoisted):
path-kernel time of a scene built with hoisting (the default) against the same scene built with B200RT_HOISTED=0.

    python scripts/hoisted_cost.py [--configs C1,C2,C3,C4,C4b,C5] [--pairs 5] [--counter-spp 64] [--out FILE.jsonl]
                                   [--bench FILE.jsonl]

Every bench.WORKLOADS config at its own resolution, spp and max depth (C2 at 1024 spp).  Both arms are resident at once,
each built with its own setting; after one warm-up of each, the two arms alternate --pairs times and the time is the
library's own CUDA-event kernel time (stats.kernel_ms).  The frames of the two arms must be the same bits.  Per arm, one
FLAG_COUNTERS render at --counter-spp gives node visits and primitive tests per ray.  With --bench, bench.py runs once
per arm (hoisting on, then B200RT_HOISTED=0) and its JSON lines go to that file.  The GPU's name and power limit are
printed with the numbers.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench import WORKLOADS  # noqa: E402
from moments_cost import gpu_identity, load_scene  # noqa: E402


def handle(rt, scene, hoisted):
    """A resident scene built with hoisting on or off (the setting is read when the scene is built)."""
    if hoisted:
        os.environ.pop("B200RT_HOISTED", None)
    else:
        os.environ["B200RT_HOISTED"] = "0"
    try:
        return rt.DeviceSceneHandle(scene)
    finally:
        os.environ.pop("B200RT_HOISTED", None)


def per_ray(rt, capi, dev, cam, spp):
    _, st = dev.render(rt.camera_with(cam, spp=spp), seed=1, flags=capi.FLAG_COUNTERS)
    return {"nodes_per_ray": round(st["node_visits"] / st["rays"], 4), "prims_per_ray": round(st["prim_tests"] / st["rays"], 4),
            "quads_per_ray": round(st["quad_tests"] / st["rays"], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--counter-spp", type=int, default=64)
    ap.add_argument("--out", default="")
    ap.add_argument("--bench", default="", help="also run bench.py once per arm; its JSON lines go to this file")
    a = ap.parse_args()
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    if rt.device_count() == 0:
        raise SystemExit("hoisted_cost.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    gpu, power = gpu_identity()
    print(f"GPU 0: {gpu}, power limit {power}, library {capi.lib()._name}", flush=True)
    rows = []
    for tag in a.configs.split(","):
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        scene = load_scene(scene_name)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=depth)
        with handle(rt, scene, True) as on, handle(rt, scene, False) as off:
            n_hoisted = on.info()["n_hoisted"]
            img_on, _ = on.render(cam, seed=1)
            img_off, _ = off.render(cam, seed=1)
            same = img_on.tobytes() == img_off.tobytes()
            t_on, t_off = [], []
            for _ in range(a.pairs):
                t_off.append(off.render(cam, seed=1)[1]["kernel_ms"])
                t_on.append(on.render(cam, seed=1)[1]["kernel_ms"])
            c_on, c_off = per_ray(rt, capi, on, cam, a.counter_spp), per_ray(rt, capi, off, cam, a.counter_spp)
            depth_on, depth_off = on.info()["tree_depth"], off.info()["tree_depth"]
        m_on, m_off = statistics.median(t_on), statistics.median(t_off)
        row = {"config": tag, "scene": scene_name, "w": w, "h": h, "spp": spp, "max_depth": depth, "n_hoisted": n_hoisted,
               "off_ms": round(m_off, 2), "on_ms": round(m_on, 2), "gain": round(m_off / m_on - 1, 4),
               "off_range_ms": [round(min(t_off), 2), round(max(t_off), 2)], "on_range_ms": [round(min(t_on), 2), round(max(t_on), 2)],
               "ranges_overlap": min(t_off) <= max(t_on) and min(t_on) <= max(t_off), "same_bits": same,
               "counters_off": c_off, "counters_on": c_on, "tree_depth_off": depth_off, "tree_depth_on": depth_on,
               "frame_sha256": hashlib.sha256(img_on.tobytes()).hexdigest()[:16], "gpu": gpu, "power_limit": power}
        rows.append(row)
        print(f"{tag:4s} {scene_name:16s} {w}x{h} {spp:5d} spp, {n_hoisted} hoisted: off {m_off:9.2f} ms [{min(t_off):.2f}, {max(t_off):.2f}]"
              f"  on {m_on:9.2f} ms [{min(t_on):.2f}, {max(t_on):.2f}]  {m_off / m_on - 1:+.2%}  {'same bits' if same else 'FRAMES DIFFER'}"
              f"  nodes/ray {c_off['nodes_per_ray']} -> {c_on['nodes_per_ray']}, prims/ray {c_off['prims_per_ray']} -> {c_on['prims_per_ray']}",
              flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if a.bench:
        with open(a.bench, "w") as f:
            for arm, env in (("on", {}), ("off", {"B200RT_HOISTED": "0"})):
                res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"], cwd=ROOT,
                                     env=dict(os.environ, **env), capture_output=True, text=True)
                line = res.stdout.strip().splitlines()[-1] if res.stdout.strip() else ""
                print(f"bench.py, hoisting {arm}: exit {res.returncode}: {line[:400]}", flush=True)
                f.write(json.dumps({"arm": arm, "returncode": res.returncode, "result": line, "stderr": res.stderr[-2000:]}) + "\n")
    if not all(r["same_bits"] for r in rows):
        raise SystemExit("hoisted_cost.py: hoisting changed a frame")


if __name__ == "__main__":
    main()
