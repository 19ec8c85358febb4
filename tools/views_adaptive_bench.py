#!/usr/bin/env python3
"""views_adaptive_bench.py — one adaptive multi-view render (rt_gpu_render_views_adaptive) against the same views
rendered adaptively one call each.

Scene: BASELINE config 4 (260 192 triangles, 32 emitters), uploaded once.  V = 8 views of 1000 x 1000: the scene camera
yawed about its own up axis, evenly over +-30 degrees (as tools/views_bench.py).  Adaptive parameters: at most 4000 spp,
min = step = 250, and a target equal to the RMS err of the uniform 1000-spp render of the same views (its err map comes
from a one-round adaptive render at min = max = 1000, as in tools/adaptive_bench.py).  Two arms on one handle, the
default max_paths_in_flight:
  batched   one render_views_adaptive call of all 8 views
  per_view  8 one-view calls render_views_adaptive([cam_v], view_base = v): rt_gpu_render_adaptive of each view
Per arm: the summed device ms of the calls (stats.render_ms), samples, ns per sample, kernel launches and rounds
(summed over the calls); best of --reps after a warm-up of both arms, the arms alternating.  The arms batch differently
(a round of 250 samples is one batch of a one-view call but several of the 8-view call, whose batches hold at most
max_paths_in_flight / (8 * 10^6) samples), so their sums may differ in the last bits and a pixel at the threshold can
stop one round apart: the fraction of pixels whose counts agree is reported.  One JSON line on stdout; the card's name,
power limit and max SM clock are part of it.

    python tools/views_adaptive_bench.py [--reps 2]
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scenes")):
    if p not in sys.path:
        sys.path.insert(0, p)

V, W, H = 8, 1000, 1000
UNIFORM_SPP, MAX_SPP, STEP = 1000, 4000, 250
SEED = 7


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def yawed(cam, degrees):
    """`cam` turned about its own up axis by `degrees` (float32)."""
    import rt_b200

    t = np.radians(degrees)
    c, s = np.float32(np.cos(t)), np.float32(np.sin(t))
    return rt_b200.Camera(cam.position, c * cam.right - s * cam.forward, cam.up, c * cam.forward + s * cam.right, cam.fov_x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    import gen_gltf
    import rt_b200  # noqa: F401
    from rt_b200 import gltf, gpu

    tmp = tempfile.mkdtemp(prefix="rt_views_adaptive_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    path = gen_gltf.generate("big_lights", tmp)
    sc = gltf.load_gltf(path, W / H)
    cams = [yawed(sc.camera(), a) for a in np.linspace(-30.0, 30.0, V)]
    result = {"metric": "adaptive multi-view render vs one adaptive call per view", "card": card(), "views": V, "width": W,
              "height": H, "max_spp": MAX_SPP, "min_step": STEP}
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_views_adaptive(cams, W, H, UNIFORM_SPP, UNIFORM_SPP, 1, 0.0, seed=SEED)  # the uniform render + err map
        uniform = g.stats()
        _, err = g.readback_adaptive()
        target = float(np.sqrt(np.mean(np.square(err[np.isfinite(err)], dtype=np.float64))))
        result["target"] = target
        result["uniform_1000spp"] = {"device_ms": uniform["render_ms"], "samples": uniform["samples"],
                                     "ns_per_sample": uniform["render_ms"] * 1e6 / uniform["samples"],
                                     "launches": uniform["kernel_launches"]}

        def rounds_of(counts):
            return int(-(-int(counts.max()) // STEP))

        def batched():
            g.render_views_adaptive(cams, W, H, MAX_SPP, STEP, STEP, target, seed=SEED)
            st = g.stats()
            counts, _ = g.readback_adaptive()
            return {"device_ms": st["render_ms"], "samples": st["samples"], "launches": st["kernel_launches"],
                    "rounds": rounds_of(counts)}, counts

        def per_view():
            row = {"device_ms": 0.0, "samples": 0, "launches": 0, "rounds": 0}
            counts = []
            for v, cam in enumerate(cams):
                g.render_views_adaptive([cam], W, H, MAX_SPP, STEP, STEP, target, seed=SEED, view_base=v)
                st = g.stats()
                c, _ = g.readback_adaptive()
                row["device_ms"] += st["render_ms"]
                row["samples"] += st["samples"]
                row["launches"] += st["kernel_launches"]
                row["rounds"] += rounds_of(c)
                counts.append(c[0])
            return row, np.stack(counts)

        arms = {"batched": batched, "per_view": per_view}
        for arm in arms.values():  # warm-up: module load, queue allocation at each shape
            arm()
        rows = {k: [] for k in arms}
        counts = {}
        for _ in range(args.reps):
            for k, arm in arms.items():
                row, counts[k] = arm()
                rows[k].append(row)
                print(json.dumps({k: row}), file=sys.stderr, flush=True)
    for k, rs in rows.items():
        best = min(rs, key=lambda r: r["device_ms"])
        result[k] = {**best, "ns_per_sample": best["device_ms"] * 1e6 / best["samples"],
                     "device_ms_all": [r["device_ms"] for r in rs]}
    result["batched_speedup_device"] = result["per_view"]["device_ms"] / result["batched"]["device_ms"]
    result["counts_agree_fraction"] = float((counts["batched"] == counts["per_view"]).mean())
    print(json.dumps(result))


if __name__ == "__main__":
    main()
