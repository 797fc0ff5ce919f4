#!/usr/bin/env python
"""Cost of the frame's tail: path-kernel time with whole tiles only (B200RT_TAIL_TILES=0) against the default chunked tail.

    python scripts/tail_cost.py [--configs C1,C2,C3,C4,C4b,C5] [--pairs 5] [--out FILE.jsonl]

Every bench.WORKLOADS config at its own resolution, spp and max depth, on one resident scene.  After one warm-up of each
arm, the two arms alternate --pairs times; the time is the library's own CUDA-event kernel time (stats.kernel_ms).  The
medians and the ranges of both arms are printed with the GPU's name and power limit.  The frames of the two arms are
compared too: the chunked tail must not change a bit.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench import WORKLOADS  # noqa: E402
from moments_cost import gpu_identity, load_scene  # noqa: E402


def render(dev, cam, tail):
    if tail is None:
        os.environ.pop("B200RT_TAIL_TILES", None)
    else:
        os.environ["B200RT_TAIL_TILES"] = tail
    try:
        img, st = dev.render(cam, seed=1)
    finally:
        os.environ.pop("B200RT_TAIL_TILES", None)
    return img, st["kernel_ms"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import cpp_raytracer_b200 as rt
    if rt.device_count() == 0:
        raise SystemExit("tail_cost.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    gpu, power = gpu_identity()
    print(f"GPU 0: {gpu}, power limit {power}", flush=True)
    rows = []
    for tag in a.configs.split(","):
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        scene = load_scene(scene_name)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=spp, max_depth=depth)
        with rt.DeviceSceneHandle(scene) as dev:
            img_whole, _ = render(dev, cam, "0")
            img_tail, _ = render(dev, cam, None)
            same = img_whole.tobytes() == img_tail.tobytes()
            whole, tail = [], []
            for _ in range(a.pairs):
                whole.append(render(dev, cam, "0")[1])
                tail.append(render(dev, cam, None)[1])
        mw, mt = statistics.median(whole), statistics.median(tail)
        row = {"config": tag, "scene": scene_name, "w": w, "h": h, "spp": spp, "max_depth": depth,
               "whole_tiles_ms": round(mw, 2), "tail_ms": round(mt, 2), "gain": round(mw / mt - 1, 4),
               "whole_tiles_range_ms": [round(min(whole), 2), round(max(whole), 2)], "tail_range_ms": [round(min(tail), 2), round(max(tail), 2)],
               "ranges_overlap": min(whole) <= max(tail), "same_bits": same,
               "frame_sha256": hashlib.sha256(img_tail.tobytes()).hexdigest()[:16], "gpu": gpu, "power_limit": power}
        rows.append(row)
        print(f"{tag:4s} {scene_name:16s} {w}x{h} {spp:5d} spp: whole tiles {mw:9.2f} ms [{min(whole):.2f}, {max(whole):.2f}]"
              f"  chunked tail {mt:9.2f} ms [{min(tail):.2f}, {max(tail):.2f}]  {mw / mt - 1:+.2%}"
              f"  {'same bits' if same else 'FRAMES DIFFER'}", flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")
    if not all(r["same_bits"] for r in rows):
        raise SystemExit("tail_cost.py: the chunked tail changed a frame")


if __name__ == "__main__":
    main()
