#!/usr/bin/env python3
"""views_bench.py — one multi-view render (rt_gpu_render_views) against the same views rendered one call each.

Scene: BASELINE config 4 (260 192 triangles, 32 emitters), uploaded once.  View v is the scene camera yawed about its
own up axis, evenly over +-30 degrees.  Two workloads:
  a  64 views of 256 x 256 at 16 spp (1 Mi paths per view: a single view leaves the GPU short of work)
  b   4 views of 1000 x 1000 at 250 spp (config 4's 1e9 samples)
Two arms per workload, on one handle: "batched" = one render_views call of all views; "per_view" = consecutive
one-view calls with view_base = v (the same frames, see rt_gpu.h).  Per arm: the summed device ms of the calls
(stats.render_ms), the host wall time around the calls and around calls + readback of the means, Msamples/s on the
device time and the kernel launches; best of --reps after a warm-up of both arms, the arms alternating.  Both arms
use the default max_paths_in_flight.  The two arms' images must be bit-identical when they run in the same batches:
in workload a every call is one batch; in workload b the 1e9 paths do not fit one batch, so the check renders it
once more with max_paths_in_flight set per arm to batches of 125 spp.  One JSON line on stdout; the card's name,
power limit and max SM clock are part of it.

    python tools/views_bench.py [--workloads a,b] [--reps 3]
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scenes")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {"a": (64, 256, 256, 16), "b": (4, 1000, 1000, 250)}  # views, width, height, spp
SEED = 7
CHECK_SPP_PER_BATCH = 125  # workload b's identity check: both arms in batches of 125 spp


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
    ap.add_argument("--workloads", default="a,b")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import gen_gltf
    import rt_b200  # noqa: F401
    from rt_b200 import gltf, gpu

    tmp = tempfile.mkdtemp(prefix="rt_views_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    path = gen_gltf.generate("big_lights", tmp)
    result = {"metric": "multi-view render vs one call per view", "card": card(), "workloads": {}}
    sc = gltf.load_gltf(path, 1.0)  # every workload is square: the same scene camera
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        for name in args.workloads.split(","):
            V, w, h, spp = WORKLOADS[name]
            cams = [yawed(sc.camera(), a) for a in np.linspace(-30.0, 30.0, V)]

            def batched(paths=0, keep=False):
                g.render_views(cams, w, h, spp, seed=SEED, max_paths_in_flight=paths)
                st = g.stats()
                return st["render_ms"], st["kernel_launches"], st["samples"], g.readback()[0] if keep else None

            def per_view(paths=0, keep=False):
                ms = launches = samples = 0
                imgs = []
                for v, cam in enumerate(cams):
                    g.render_views([cam], w, h, spp, seed=SEED, view_base=v, max_paths_in_flight=paths)
                    st = g.stats()
                    ms, launches, samples = ms + st["render_ms"], launches + st["kernel_launches"], samples + st["samples"]
                    if keep:
                        imgs.append(g.readback()[0][0])
                return ms, launches, samples, np.stack(imgs) if keep else None

            def timed(arm, **kw):
                t0 = time.perf_counter()
                out = arm(**kw)
                return out, (time.perf_counter() - t0) * 1e3

            arms = {"batched": batched, "per_view": per_view}
            for arm in arms.values():  # warm-up: module load, queue allocation at each shape
                arm(keep=True)
            rows = {k: [] for k in arms}
            images = {}
            for _ in range(args.reps):
                for k, arm in arms.items():
                    (ms, launches, samples, _), wall = timed(arm)
                    (_, _, _, images[k]), wall_rb = timed(arm, keep=True)
                    rows[k].append({"device_ms": ms, "wall_ms": wall, "wall_with_readback_ms": wall_rb, "launches": launches,
                                    "samples": samples})
            if name == "b":  # the identity check in equal batches (workload a: every call is already one batch)
                per = w * h * CHECK_SPP_PER_BATCH
                images = {"batched": batched(V * per, keep=True)[3], "per_view": per_view(per, keep=True)[3]}
            summary = {}
            for k, rs in rows.items():
                best = min(rs, key=lambda r: r["device_ms"])
                summary[k] = {"device_ms": best["device_ms"], "wall_ms": min(r["wall_ms"] for r in rs),
                              "wall_with_readback_ms": min(r["wall_with_readback_ms"] for r in rs),
                              "msamples_per_s": best["samples"] / best["device_ms"] * 1e-3, "launches": best["launches"],
                              "samples": best["samples"], "device_ms_all": [r["device_ms"] for r in rs]}
            summary["batched_speedup_device"] = summary["per_view"]["device_ms"] / summary["batched"]["device_ms"]
            summary["batched_speedup_wall"] = summary["per_view"]["wall_with_readback_ms"] / summary["batched"]["wall_with_readback_ms"]
            same = bool(np.array_equal(images["batched"], images["per_view"]))
            result["workloads"][name] = {"views": V, "width": w, "height": h, "spp": spp, "images_bit_identical": same, **summary}
            print(json.dumps({name: result["workloads"][name]}), file=sys.stderr, flush=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
