#!/usr/bin/env python
"""A/B of two builds of the library: path-kernel time of every benchmark config, one subprocess per run.

    python scripts/slab_pairs_cost.py LIB_A LIB_B [--names parent,paired] [--configs C1,C2,C3,C4,C4b,C5] [--pairs 5]
                                      [--out FILE.jsonl]

Written for the node step's paired FP32 slab tests (FFMA2 / FMUL2) against the scalar form, and usable for any two
builds of the same ABI.  Each run is a fresh process that loads its library through B200RT_LIB and renders every
bench.WORKLOADS config at its own resolution, spp and max depth: one warm-up render, then one timed render; the time
is the library's own CUDA-event kernel time (stats.kernel_ms).  The runs alternate A B, B A, A B, ... for --pairs
pairs, and per config the medians and ranges of both libraries are printed with the GPU's name, power limit and SM
clocks read in the same call.  The first run of each library also records the traversal counters (node visits and
primitive tests per ray, 16 spp) and every run the SHA-256 of its HDR frame: the two builds must agree on both.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import WORKLOADS  # noqa: E402


def gpu_identity():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            name, power, sm, sm_max = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
            return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}
    except (OSError, subprocess.SubprocessError, ValueError):
        pass
    return {"gpu": "unknown", "power_limit": "unknown", "sm_clock": "unknown", "sm_clock_max": "unknown"}


def load_scene(name, cache_dir):
    """The golden dump, or host/b200rt_scenes' dump of the multi-million-primitive scenes (made once per A/B, in
    cache_dir), as bench.py loads them."""
    from cpp_raytracer_b200 import build, scene_io
    golden = os.path.join(ROOT, "tests", "golden", f"{name}.scene.gz")
    if os.path.exists(golden):
        return scene_io.load_scene(golden)
    path = os.path.join(cache_dir, f"{name}.scene")
    if not os.path.exists(path):
        subprocess.run([build.build_host(), name, "dump", path], check=True, capture_output=True)
    return scene_io.load_scene(path)


def worker(configs, cache_dir, counters):
    """One run: every config with the library B200RT_LIB names; one JSON line per config on stdout."""
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    if rt.device_count() == 0:
        raise SystemExit("slab_pairs_cost.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    for tag in configs:
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        scene = load_scene(scene_name, cache_dir)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=depth)
        with rt.DeviceSceneHandle(scene) as dev:
            dev.render(cam, seed=1)
            img, st = dev.render(cam, seed=1)
            row = {"config": tag, "kernel_ms": st["kernel_ms"], "frame_sha256": hashlib.sha256(img.tobytes()).hexdigest()}
            if counters:
                _, sc = dev.render(rt.camera_with(cam, spp=min(spp, 16)), seed=1, flags=capi.FLAG_COUNTERS)
                row["node_visits_per_ray"] = sc["node_visits"] / max(1, sc["rays"])
                row["prim_tests_per_ray"] = sc["prim_tests"] / max(1, sc["rays"])
        print(json.dumps(row), flush=True)


def run(lib, configs, cache_dir, counters):
    env = dict(os.environ, B200RT_LIB=os.path.abspath(lib))
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--configs", ",".join(configs), "--cache-dir", cache_dir]
    if counters:
        cmd.append("--counters")
    res = subprocess.run(cmd, env=env, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise SystemExit(f"slab_pairs_cost.py: the run with {lib} failed")
    return {r["config"]: r for r in (json.loads(x) for x in res.stdout.splitlines() if x.startswith("{"))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*", help="LIB_A LIB_B")
    ap.add_argument("--names", default="a,b")
    ap.add_argument("--configs", default=",".join(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--out", default="")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--cache-dir", default="", help=argparse.SUPPRESS)
    ap.add_argument("--counters", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    configs = a.configs.split(",")
    if a.worker:
        worker(configs, a.cache_dir, a.counters)
        return
    if len(a.libs) != 2:
        raise SystemExit("slab_pairs_cost.py: give two library paths")
    names = a.names.split(",")
    ident = gpu_identity()
    print(f"GPU 0: {ident['gpu']}, power limit {ident['power_limit']}, SM clock {ident['sm_clock']} "
          f"(max {ident['sm_clock_max']})", flush=True)
    runs = {0: [], 1: []}
    with tempfile.TemporaryDirectory() as cache_dir:
        for p in range(a.pairs):
            for k in ((0, 1) if p % 2 == 0 else (1, 0)):
                runs[k].append(run(a.libs[k], configs, cache_dir, counters=(p == 0)))
    rows = []
    for tag in configs:
        ta, tb = [[r[tag]["kernel_ms"] for r in runs[k]] for k in (0, 1)]
        ma, mb = statistics.median(ta), statistics.median(tb)
        same_bits = len({r[tag]["frame_sha256"] for k in (0, 1) for r in runs[k]}) == 1
        cnt = [next(r[tag] for r in runs[k] if "node_visits_per_ray" in r[tag]) for k in (0, 1)]
        same_counters = all(cnt[0][f] == cnt[1][f] for f in ("node_visits_per_ray", "prim_tests_per_ray"))
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        row = {"config": tag, "scene": scene_name, "w": w, "h": h, "spp": spp, "max_depth": depth, "pairs": a.pairs,
               f"{names[0]}_ms": round(ma, 2), f"{names[1]}_ms": round(mb, 2), "gain": round(ma / mb - 1, 4),
               f"{names[0]}_range_ms": [round(min(ta), 2), round(max(ta), 2)],
               f"{names[1]}_range_ms": [round(min(tb), 2), round(max(tb), 2)],
               "ranges_overlap": not (max(ta) < min(tb) or max(tb) < min(ta)), "same_bits": same_bits,
               "node_visits_per_ray": round(cnt[1]["node_visits_per_ray"], 4),
               "prim_tests_per_ray": round(cnt[1]["prim_tests_per_ray"], 4), "same_counters": same_counters,
               "frame_sha256": runs[1][0][tag]["frame_sha256"][:16], **ident}
        rows.append(row)
        print(f"{tag:4s} {scene_name:16s} {w}x{h} {spp:5d} spp: {names[0]} {ma:9.2f} ms [{min(ta):.2f}, {max(ta):.2f}]"
              f"  {names[1]} {mb:9.2f} ms [{min(tb):.2f}, {max(tb):.2f}]  {ma / mb - 1:+.2%}"
              f"  {'ranges apart' if not row['ranges_overlap'] else 'ranges overlap'}"
              f"  {'same bits' if same_bits else 'FRAMES DIFFER'}  {'same counters' if same_counters else 'COUNTERS DIFFER'}",
              flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not all(r["same_bits"] and r["same_counters"] for r in rows):
        raise SystemExit("slab_pairs_cost.py: the two libraries disagree on a frame or on the traversal counters")


if __name__ == "__main__":
    main()
