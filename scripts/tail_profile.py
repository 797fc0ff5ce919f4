#!/usr/bin/env python
"""The frame's tail, measured: when every block of the path kernel starts and ends, and how much of the GPU's block slots
the frame leaves idle.

    python scripts/tail_profile.py [--configs C1,C2,C3,C5] [--tails 0,default] [--out FILE.jsonl]

Runs the diagnostic build (-DB200RT_BLOCK_TIMES, scratch_libs/libb200rt_blocktimes.so, built here if missing), in which
thread 0 of every path_megakernel_pool block records %globaltimer at its start and end and its SM.  For each config at its
bench size and each tail setting (B200RT_TAIL_TILES value, "default" = the library's own plan) it renders one frame after a
warm-up and reports:
  slots       resident path blocks at once: the most blocks seen running together
  span        first block start to last block end
  idle share  1 - sum(block durations) / (slots x span): the share of block-slot time no block used
  drain       last block start to last block end: how long the frame ran without a block waiting to start
  curve       resident blocks against time, in 40 steps of the span
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
DIAG_LIB = os.path.join(ROOT, "scratch_libs", "libb200rt_blocktimes.so")


def block_stats(t, steps=40):
    import numpy as np
    t = t[t[:, 1] > 0]
    start, end = t[:, 0].astype(np.int64), t[:, 1].astype(np.int64)
    t0, t1 = int(start.min()), int(end.max())
    ev = np.concatenate([np.stack([start, np.ones_like(start)], 1), np.stack([end, -np.ones_like(end)], 1)])
    ev = ev[np.lexsort((ev[:, 1], ev[:, 0]))]                      # ends before starts at equal times
    level = np.cumsum(ev[:, 1])
    slots = int(level.max())
    span = t1 - t0
    grid = t0 + (np.arange(steps) + 0.5) * span / steps
    curve = [int(level[max(0, np.searchsorted(ev[:, 0], g, side="right") - 1)]) for g in grid]
    return {"blocks": int(len(t)), "sms": int(len(np.unique(t[:, 2]))), "slots": slots, "span_ms": span / 1e6,
            "idle_share": 1.0 - float((end - start).sum()) / (slots * span), "drain_ms": (t1 - int(start.max())) / 1e6,
            "block_ms_median": float(np.median(end - start)) / 1e6, "curve": curve}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C1,C2,C3,C5")
    ap.add_argument("--tails", default="0,default")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not os.path.exists(DIAG_LIB):
        from cpp_raytracer_b200 import build
        build.build_variant("blocktimes", ["-DB200RT_BLOCK_TIMES"])
    os.environ["B200RT_LIB"] = DIAG_LIB
    import ctypes
    import torch
    import cpp_raytracer_b200 as rt
    from cpp_raytracer_b200 import capi
    from bench import WORKLOADS
    from moments_cost import gpu_identity, load_scene
    if rt.device_count() == 0:
        raise SystemExit("tail_profile.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    arm = capi.lib().b200rt_debug_block_times
    arm.argtypes, arm.restype = [ctypes.c_void_p, ctypes.c_uint64], ctypes.c_int
    gpu, power = gpu_identity()
    print(f"GPU 0: {gpu}, power limit {power}", flush=True)
    rows = []
    for tag in a.configs.split(","):
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        scene = load_scene(scene_name)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=depth)
        tiles = ((w + 7) // 8) * ((h + 31) // 32)
        buf = torch.zeros(tiles * 10 * 3, dtype=torch.int64, device="cuda")      # room for every chunk block of any plan here
        with rt.DeviceSceneHandle(scene) as dev:
            for tail in a.tails.split(","):
                if tail == "default":
                    os.environ.pop("B200RT_TAIL_TILES", None)
                else:
                    os.environ["B200RT_TAIL_TILES"] = tail
                dev.render(rt.camera_with(cam, spp=max(1, spp // 16)), seed=1)    # warm-up
                buf.zero_()
                torch.cuda.synchronize()
                assert arm(buf.data_ptr(), tiles * 10) == 0
                _, st = dev.render(cam, seed=1)
                torch.cuda.synchronize()
                assert arm(None, 0) == 0
                s = block_stats(buf.view(-1, 3).cpu().numpy())
                s.update({"config": tag, "scene": scene_name, "w": w, "h": h, "spp": spp, "tail": tail, "tiles": tiles,
                          "kernel_ms": st["kernel_ms"], "gpu": gpu, "power_limit": power})
                rows.append(s)
                print(f"{tag:4s} tail={tail:8s} blocks {s['blocks']:6d} slots {s['slots']:4d} span {s['span_ms']:9.2f} ms  "
                      f"idle share {s['idle_share']:6.2%}  drain {s['drain_ms']:7.2f} ms  block median {s['block_ms_median']:7.2f} ms",
                      flush=True)
                print("     curve " + " ".join(str(c) for c in s["curve"]), flush=True)
        os.environ.pop("B200RT_TAIL_TILES", None)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
