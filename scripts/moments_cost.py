#!/usr/bin/env python
"""Cost of the second-moment render: Mpaths/s of DeviceSceneHandle.render and render_moments on the same resident scene.

    python scripts/moments_cost.py [--configs C1,C2,C3,C4,C4b,C5] [--spp 64] [--reps 3] [--out FILE.jsonl]

Every bench.WORKLOADS config at its own resolution and max depth, at --spp samples per pixel, plus C2 at its full spp.
After one warm-up of each, the two calls alternate --reps times on the same handle; the time is the library's own
CUDA-event kernel time (stats.kernel_ms), the figure is the median.  Scenes load as bench.py loads them: the golden dump,
or host/b200rt_scenes for the multi-million-primitive ones.  The GPU's name and power limit are printed with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import WORKLOADS  # noqa: E402


def load_scene(name):
    from cpp_raytracer_b200 import build, scene_io
    golden = os.path.join(ROOT, "tests", "golden", f"{name}.scene.gz")
    if os.path.exists(golden):
        return scene_io.load_scene(golden)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, f"{name}.scene")
        subprocess.run([build.build_host(), name, "dump", path], check=True, capture_output=True)
        return scene_io.load_scene(path)


def gpu_identity():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
            return name, power
    except (OSError, subprocess.SubprocessError):
        pass
    return "unknown", "unknown"


def measure(dev, cam, reps):
    mp = lambda st: st["paths"] / st["kernel_ms"] / 1e3   # noqa: E731  Mpaths/s
    dev.render(cam, seed=1)
    dev.render_moments(cam, seed=1)
    plain, moments = [], []
    for _ in range(reps):
        plain.append(mp(dev.render(cam, seed=1)[1]))
        moments.append(mp(dev.render_moments(cam, seed=1)[2]))
    return statistics.median(plain), statistics.median(moments), plain, moments


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(WORKLOADS))
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import cpp_raytracer_b200 as rt
    if rt.device_count() == 0:
        raise SystemExit("moments_cost.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    gpu, power = gpu_identity()
    print(f"GPU 0: {gpu}, power limit {power}")
    runs = [(tag, a.spp) for tag in a.configs.split(",")] + [("C2", WORKLOADS["C2"][3])]
    rows = []
    for tag, spp in runs:
        scene_name, w, h, _, depth = WORKLOADS[tag][:5]
        scene = load_scene(scene_name)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=depth)
        with rt.DeviceSceneHandle(scene) as dev:
            p, m, ps, ms = measure(dev, cam, a.reps)
        row = {"config": tag, "scene": scene_name, "w": w, "h": h, "spp": spp, "max_depth": depth,
               "render_mpaths_s": round(p, 1), "render_moments_mpaths_s": round(m, 1), "moments_vs_render": round(m / p, 4),
               "render_runs": [round(x, 1) for x in ps], "moments_runs": [round(x, 1) for x in ms], "gpu": gpu, "power_limit": power}
        rows.append(row)
        print(f"{tag:4s} {scene_name:16s} {w}x{h} {spp:5d} spp depth {depth:4d}: render {p:8.1f}  render_moments {m:8.1f} Mpaths/s"
              f"  ({m / p - 1:+.1%})", flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
