#!/usr/bin/env python
"""Generates the committed golden fixtures FROM THE REFERENCE ITSELF (oracle/_ref/ref_bridge =
the unmodified reference headers compiled in this container, see oracle/Makefile).

    python tests/golden/make_golden.py            # needs oracle/_ref/ref_bridge

For every small scene it writes under tests/golden/:
    <scene>.scene.gz        flat dump of the reference-built Scene + Camera (incl. what
                            Camera::init derives)  -> pins scene builders and b200rt_camera_init
    <scene>.rays.gz         fixed ray set: camera rays (fixed jitter table), rays recorded from the
                            reference's own paths (all bounces), adversarial rays
    <scene>.hits.gz         the reference's (prim, t) for those rays through BVH::hit_by semantics
    <scene>.hits_brute.gz   same through Scene::hit_by (brute force)  [small scenes only]
    <scene>.refA.npy.gz / <scene>.refB.npy.gz
                            two statistically independent reference renders (float32 linear HDR)
                            at reduced resolution -> image-convergence tests and their noise floor
    <scene>.render1t.npz    single-threaded reference render in exact doubles + the LCG state it started
                            from -> BIT-EXACT pin of the C restatement's whole path loop
    kat.json                unit known answers (LCG stream, reflect/refract/Schlick, tone map)
The big scenes (raining: 2.2 M quads, millions_lights: 3.1 M spheres) are NOT committed; where the
bridge binary is built, the live-reference tests regenerate them with it.  tests/golden/make_big_golden.py
stores a digest and a ray sample of them for the tests that run without it.
"""
import gzip
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from cpp_raytracer_b200 import scene_io  # noqa: E402

BRIDGE = os.path.join(ROOT, "oracle", "_ref", "ref_bridge")

# scene -> (render w, h, spp for the reference renders; depth override or None)
SCENES = {
    "rtow_final": (160, 90, 1024, None),
    "rtow_lights": (160, 90, 2048, None),
    "quads": (96, 96, 512, None),
    "cornell_empty": (96, 96, 1024, 50),
    "cornell": (96, 96, 2048, 50),
    "xmas": (160, 90, 2048, None),
    "pathological": (0, 0, 0, None),
}
N_CAMERA, N_RECORDED = 2048, 2048


def run(args, **kw):
    res = subprocess.run([BRIDGE, *args], capture_output=True, text=True, **kw)
    if res.returncode != 0:
        raise RuntimeError(f"ref_bridge {' '.join(args)} failed:\n{res.stdout}\n{res.stderr}")
    return [json.loads(l) for l in res.stdout.splitlines() if l.startswith("{")]


def gz_copy(src, dst):
    with open(src, "rb") as f, gzip.GzipFile(dst, "wb", mtime=0) as g:
        g.write(f.read())


def adversarial_rays(scene, rng):
    """Rays chosen to stress the precision design: axis-parallel directions (zero components,
    signed zeros), grazing rays tangent to spheres, origins inside / on primitives, huge and
    tiny direction magnitudes, far-field rays on the big ground primitive."""
    rays = []
    sph, quads = scene.spheres, scene.quads
    cam = scene.camera[0]
    c0 = cam["center"]
    targets = []
    if len(sph):
        pick = rng.choice(len(sph), size=min(64, len(sph)), replace=False)
        for i in pick:
            c, r = sph["c"][i], sph["r"][i]
            targets.append(c)
            # axis-parallel through the centre and exactly tangent
            for ax in range(3):
                d = np.zeros(3); d[ax] = 1.0
                rays.append(np.concatenate([c - 3 * abs(r) * d - 0.0, d]))
                rays.append(np.concatenate([c + 3 * abs(r) * d, -d]))
                off = np.zeros(3); off[(ax + 1) % 3] = r          # tangent line
                rays.append(np.concatenate([c - 3 * abs(r) * d + off, d]))
                off2 = np.zeros(3); off2[(ax + 1) % 3] = r * (1 - 1e-12)
                rays.append(np.concatenate([c - 3 * abs(r) * d + off2, d]))
            # from inside the sphere, random direction (must find the far root)
            d = rng.normal(size=3)
            rays.append(np.concatenate([c + 0.3 * r * d / np.linalg.norm(d), rng.normal(size=3)]))
            # grazing from the camera: aim at the silhouette
            v = c - c0
            dist = np.linalg.norm(v)
            if dist > abs(r):
                perp = np.cross(v, rng.normal(size=3)); perp /= np.linalg.norm(perp)
                for eps in (-1e-9, 0.0, 1e-9, 1e-6):
                    rays.append(np.concatenate([c0, v + perp * abs(r) * (1 + eps) * dist / np.sqrt(dist**2 - r**2)]))
            # origin exactly on the surface, direction leaving / entering
            n = rng.normal(size=3); n /= np.linalg.norm(n)
            p = c + r * n
            rays.append(np.concatenate([p, n + 0.5 * rng.normal(size=3)]))
            rays.append(np.concatenate([p, -n + 0.5 * rng.normal(size=3)]))
    if len(quads):
        pick = rng.choice(len(quads), size=min(32, len(quads)), replace=False)
        for i in pick:
            v, s1, s2 = quads["v"][i], quads["s1"][i], quads["s2"][i]
            n = np.cross(s1, s2)
            nn = n / np.linalg.norm(n)
            ctr = v + 0.5 * s1 + 0.5 * s2
            targets.append(ctr)
            L = max(np.linalg.norm(s1), np.linalg.norm(s2))
            for a, b in ((0.5, 0.5), (0.0, 0.0), (1.0, 1.0), (0.0, 0.5), (1.0, 0.25), (1 + 1e-12, 0.5), (-1e-12, 0.5)):
                p = v + a * s1 + b * s2            # centre, corners, edges, just outside
                rays.append(np.concatenate([p + nn * L, -nn]))
                rays.append(np.concatenate([p - nn * 0.25 * L, nn * 3.0]))
            rays.append(np.concatenate([ctr + nn * L, s1]))            # parallel to the plane
            rays.append(np.concatenate([ctr + nn * L, s1 - 1e-10 * nn]))  # almost parallel (|den| < 1e-9 cut)
            rays.append(np.concatenate([ctr, nn]))                     # origin in the plane
    targets = np.array(targets) if targets else np.zeros((1, 3))
    # scaled directions (rays are never normalised in the reference)
    for k in range(64):
        t = targets[rng.integers(len(targets))]
        d = t - c0 + 0.05 * rng.normal(size=3)
        rays.append(np.concatenate([c0, d * 1e6]))
        rays.append(np.concatenate([c0, d * 1e-6]))
        rays.append(np.concatenate([c0, np.where(np.abs(d) < 0.3 * np.abs(d).max(), -0.0, d)]))  # signed zeros
    # far field: from high above, shallow angles towards the horizon (big ground primitive)
    for k in range(128):
        ang = rng.uniform(0, 2 * np.pi)
        elev = -10 ** rng.uniform(-6, -1)
        o = c0 + np.array([0, rng.uniform(0, 50), 0])
        rays.append(np.concatenate([o, [np.cos(ang), elev, np.sin(ang)]]))
    # pure axis directions from random origins near the camera
    for ax in range(3):
        for sgn in (1.0, -1.0):
            for k in range(16):
                d = np.zeros(3); d[ax] = sgn
                rays.append(np.concatenate([c0 + rng.normal(size=3) * 5, d]))
    return np.array(rays, dtype=np.float64)


# single-threaded double-precision renders for the BIT-EXACT pin of the C restatement
RENDER_1T = {"rtow_final": (24, 16, 4, 20), "rtow_lights": (24, 16, 4, 20), "quads": (16, 16, 4, 50),
             "cornell": (16, 16, 4, 50), "xmas": (24, 16, 2, 50)}


def make_render1t(tmp):
    for name, (w, h, spp, depth) in RENDER_1T.items():
        out = os.path.join(tmp, f"{name}.f64")
        lines = run([name, "--w", str(w), "--h", str(h), "--spp", str(spp), "--depth", str(depth), "--threads", "1",
                     "lcg_state", "render_f64", out])
        state = lines[0]["state_after_this_draw"]
        img = scene_io.load_hdr(out)
        assert img.dtype == np.float64
        np.savez_compressed(os.path.join(HERE, f"{name}.render1t.npz"), image=img, lcg_state=np.uint32(state),
                            w=w, h=h, spp=spp, max_depth=depth)
        print("render1t", name, state, flush=True)


def main():
    if not os.path.exists(BRIDGE):
        sys.exit("build oracle/_ref/ref_bridge first (make -C oracle ref)")
    tmp = tempfile.mkdtemp(prefix="golden_")
    part = sys.argv[1] if len(sys.argv) > 1 else "all"
    if part in ("all", "render1t"):
        make_render1t(tmp)
    if part in ("all", "kat"):
        run(["cornell_empty", "kat", os.path.join(HERE, "kat.json")])
    if part != "all":
        return
    summary = {}
    for name, (w, h, spp, depth) in SCENES.items():
        rng = np.random.default_rng(abs(hash(name)) % (2**32) if False else sum(map(ord, name)))
        sc_path = os.path.join(tmp, f"{name}.scene")
        rec_path = os.path.join(tmp, f"{name}.rec")
        rec_opts = ["--w", "64", "--h", "36", "--spp", "8", "--threads", "1"] if name != "pathological" else []
        cmds = ["dump", sc_path]
        if name != "pathological":
            cmds += ["record", str(N_RECORDED), "5", rec_path]
        # NB: options change the camera that `dump` writes; dump the scene with its own camera first
        run([name, "dump", sc_path])
        scene = scene_io.load_scene(sc_path)
        parts = [scene_io.camera_rays(scene.camera, N_CAMERA, seed=7)]
        if name != "pathological":
            run([name, *rec_opts, "record", str(N_RECORDED), "5", rec_path])
            rec, _, _ = scene_io.load_rays(rec_path)
            parts.append(rec)
        parts.append(adversarial_rays(scene, rng))
        rays = np.concatenate(parts, axis=0)
        rays_path = os.path.join(tmp, f"{name}.rays")
        scene_io.save_rays(rays_path, rays, 1e-5, float("inf"))
        hits_path = os.path.join(tmp, f"{name}.hits")
        brute_path = os.path.join(tmp, f"{name}.hits_brute")
        out = run([name, "raycast", rays_path, hits_path, "raycast", rays_path, brute_path, "brute"])
        gz_copy(sc_path, os.path.join(HERE, f"{name}.scene.gz"))
        gz_copy(rays_path, os.path.join(HERE, f"{name}.rays.gz"))
        gz_copy(hits_path, os.path.join(HERE, f"{name}.hits.gz"))
        gz_copy(brute_path, os.path.join(HERE, f"{name}.hits_brute.gz"))
        prim, t = scene_io.load_hits(hits_path)
        primb, tb = scene_io.load_hits(brute_path)
        summary[name] = {"rays": int(len(rays)), "hit_frac": float((prim >= 0).mean()),
                         "bvh_vs_brute_id_mismatch": int((prim != primb).sum()),
                         "bvh_vs_brute_t_mismatch": int((t != tb).sum()), "raycast": out}
        if w:
            for tag, rs in (("refA", 101), ("refB", 202)):
                hdr_path = os.path.join(tmp, f"{name}.{tag}.hdr")
                opts = ["--w", str(w), "--h", str(h), "--spp", str(spp), "--render-seed", str(rs)]
                if depth:
                    opts += ["--depth", str(depth)]
                info = run([name, *opts, "render", hdr_path])[-1]
                img = scene_io.load_hdr(hdr_path).astype(np.float32)
                with gzip.GzipFile(os.path.join(HERE, f"{name}.{tag}.npy.gz"), "wb", mtime=0) as g:
                    np.save(g, img)
                summary[name][tag] = {k: info[k] for k in ("w", "h", "spp", "max_depth", "seconds")}
        print(name, json.dumps(summary[name])[:300], flush=True)
    with open(os.path.join(HERE, "golden_summary.json"), "w") as f:
        json.dump(summary, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
