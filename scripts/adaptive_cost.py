#!/usr/bin/env python
"""What adaptive sampling buys: time to a given image quality against uniform sampling, per benchmark config.

    python scripts/adaptive_cost.py [--configs C1,C2,C3,C4,C4b,C5] [--max-spp N] [--ref-factor 4] [--out FILE.jsonl]

Every bench.WORKLOADS config at its own resolution and max depth, with a maximum of the config's spp (or --max-spp, if
smaller) samples per pixel, min_spp = max/16 and step_spp = max/16.  The target: a uniform render at max/4 samples gives each pixel's
ratio r = err / level (b200rt.h); a pixel's ratio falls as 1/sqrt(n), so rel_noise = the 90th percentile of r x
sqrt((max/4) / max) lets about the noisiest tenth of the pixels run to the maximum.  Reported per config:
  - adaptive: total paths, passes, path-kernel and decision-kernel time (torch.profiler, CUDA activities, in a run of
    their own), the library's device span (stats.kernel_ms: first kernel to last, so it includes the host round trip
    after every pass) and the wall time of the call (median of --reps);
  - the RMSE of the adaptive image and of a uniform render with the same total path count against a uniform reference
    of --ref-factor x max samples with another seed (the reference's own noise is part of both figures);
  - the uniform spp that reaches the adaptive RMSE (RMSE x sqrt(n) is about constant; two refinements), with its wall time.
Scenes load as bench.py loads them.  The GPU's name and power limit are printed and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

from bench import WORKLOADS  # noqa: E402
from moments_cost import gpu_identity, load_scene  # noqa: E402

SEED, REF_SEED = 1, 0x5EED


def ratio(mean, m2, n):
    """err / level of every pixel with level > 0, by the rule of b200rt_render_adaptive."""
    mean = mean.astype(np.float64)
    m2 = m2.astype(np.float64)
    d = m2 - mean * mean
    var = np.where(d <= m2 * 2.0 ** -20 + 2.0 ** -24, 0.0, (n / (n - 1)) * d)
    err = np.sqrt(var.sum(axis=-1) / (3.0 * n))
    level = mean.mean(axis=-1)
    ok = level > 0
    return err[ok] / level[ok]


def rmse(img, ref):
    return float(np.sqrt(np.mean((img.astype(np.float64) - ref.astype(np.float64)) ** 2)))


def timed(fn, reps):
    fn()
    walls, outs = [], None
    for _ in range(reps):
        t = time.perf_counter()
        outs = fn()
        walls.append((time.perf_counter() - t) * 1e3)
    return statistics.median(walls), outs


def kernel_times(fn):
    """Device time per kernel family of one call of fn, from torch.profiler's CUDA activity records."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    fam = {"path": 0.0, "decision": 0.0, "other": 0.0}
    n_path = 0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "path_megakernel_pool" in ev.name:
            fam["path"] += us; n_path += 1
        elif "adaptive_" in ev.name:
            fam["decision"] += us
        else:
            fam["other"] += us
    return {k: v / 1e3 for k, v in fam.items()}, n_path


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default=",".join(WORKLOADS))
    ap.add_argument("--max-spp", type=int, default=0)
    ap.add_argument("--ref-factor", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import cpp_raytracer_b200 as rt
    if rt.device_count() == 0:
        raise SystemExit("adaptive_cost.py: no CUDA device (this measures the GPU; there is nothing to measure without one)")
    gpu, power = gpu_identity()
    print(f"GPU 0: {gpu}, power limit {power}", flush=True)
    rows = []
    for tag in a.configs.split(","):
        scene_name, w, h, spp, depth = WORKLOADS[tag][:5]
        mx = min(spp, a.max_spp) if a.max_spp > 0 else spp
        step = max(2, mx // 16)
        scene = load_scene(scene_name)
        cam = rt.camera_with(scene.camera, image_w=w, image_h=h, spp=mx, max_depth=depth)
        px = w * h
        with rt.DeviceSceneHandle(scene) as dev:
            n0 = max(2, mx // 4)
            m, q, _ = dev.render_moments(cam, seed=SEED, sample_count=n0)
            rel = float(np.quantile(ratio(m, q, n0), 0.9)) * math.sqrt(n0 / mx)
            run = lambda: dev.render_adaptive(cam, rel, min_spp=step, step_spp=step, seed=SEED)  # noqa: E731
            wall_a, (img_a, _, spp_a, st_a) = timed(run, a.reps)
            fam, passes = kernel_times(run)
            paths = int(st_a["paths"])
            n_eq = max(1, round(paths / px))
            ref, _ = dev.render(cam, seed=REF_SEED, sample_count=a.ref_factor * mx)
            r_a = rmse(img_a, ref)
            uni = lambda n: dev.render(cam, seed=SEED, sample_count=n)  # noqa: E731
            r_eq = rmse(uni(n_eq)[0], ref)
            # the uniform spp with RMSE r_a: RMSE^2 = c / n + ref noise; fit on two points, then check
            n_need, r_need = n_eq, r_eq
            for _ in range(2):
                n_next = max(1, min(1 << 16, round(n_need * (r_need / r_a) ** 2)))
                if n_next == n_need:
                    break
                n_need, r_need = n_next, rmse(uni(n_next)[0], ref)
            wall_u, (_, st_u) = timed(lambda: uni(n_need), a.reps)
        hist = {int(k): int(v) for k, v in zip(*np.unique(spp_a, return_counts=True))}
        row = {"config": tag, "scene": scene_name, "w": w, "h": h, "max_spp": mx, "min_spp": step, "step_spp": step,
               "rel_noise": rel, "adaptive_paths": paths, "adaptive_mean_spp": paths / px, "passes": passes,
               "path_kernel_ms": round(fam["path"], 3), "decision_kernel_ms": round(fam["decision"], 3),
               "other_kernel_ms": round(fam["other"], 3), "adaptive_device_span_ms": round(st_a["kernel_ms"], 3),
               "adaptive_wall_ms": round(wall_a, 3), "spp_histogram": hist,
               "ref_spp": a.ref_factor * mx, "rmse_adaptive": r_a, "uniform_same_paths_spp": n_eq, "rmse_uniform_same_paths": r_eq,
               "uniform_spp_for_same_rmse": n_need, "rmse_uniform_at_that_spp": r_need,
               "uniform_kernel_ms": round(st_u["kernel_ms"], 3), "uniform_wall_ms": round(wall_u, 3),
               "wall_speedup": round(wall_u / wall_a, 3), "gpu": gpu, "power_limit": power}
        rows.append(row)
        if a.out:
            with open(a.out, "w") as f:
                for r in rows:
                    f.write(json.dumps(r) + "\n")
        print(f"{tag:4s} {scene_name:16s} {w}x{h} max {mx:4d}: adaptive {paths / px:7.1f} spp/px in {passes} passes, path {fam['path']:8.1f} ms, "
              f"decision {fam['decision']:6.2f} ms, wall {wall_a:8.1f} ms, RMSE {r_a:.4g} | uniform {n_eq} spp RMSE {r_eq:.4g}; "
              f"{n_need} spp for RMSE {r_need:.4g}: wall {wall_u:8.1f} ms  (x{wall_u / wall_a:.2f})", flush=True)


if __name__ == "__main__":
    main()
