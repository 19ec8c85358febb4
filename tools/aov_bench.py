#!/usr/bin/env python3
"""aov_bench.py — the cost of the AOV render (rt_gpu_render_aov) against the beauty render.

Scene: BASELINE config 4 (260 192 triangles, 32 emitters, 1000 x 1000), uploaded once, the scene camera.  Arms,
alternating, best of --reps after a warm-up of every arm:
  beauty      rt_gpu_render at --beauty-spp (250: the reference point)
  aov_<n>     rt_gpu_render_aov at n spp for n in --aov-spp (1, 16, 64)
Per arm: device ms (stats.render_ms), ns per sample, extension rays per sample and the kernel launches.  Per AOV arm also
the paths of one batch and the bytes a batch holds: the beauty queues (140 B per path) plus the AOV slots (48 B per
path), from the library's batch rule (max_paths_in_flight = 0: up to 512 Mi paths, at most half the free memory).
One JSON line on stdout; the card's name, power limit and max SM clock are part of it.

    python tools/aov_bench.py [--reps 3] [--beauty-spp 250] [--aov-spp 1,16,64]
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scenes")):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 7
QUEUE_BYTES, AOV_BYTES = 140, 48  # per path: rt_gpu.cu kBytesPerPath, kAovBytesPerPath


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--beauty-spp", type=int, default=250)
    ap.add_argument("--aov-spp", default="1,16,64")
    ap.add_argument("--size", type=int, default=1000)
    args = ap.parse_args()
    import gen_gltf
    from rt_b200 import gltf, gpu

    tmp = tempfile.mkdtemp(prefix="rt_aov_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    sc = gltf.load_gltf(gen_gltf.generate("big_lights", tmp), 1.0)
    w = h = args.size
    aov_spp = [int(x) for x in args.aov_spp.split(",")]
    result = {"metric": "AOV render cost against the beauty render", "card": card(), "scene": "config 4 (big_lights)", "width": w,
              "height": h, "beauty_spp": args.beauty_spp, "arms": {}}
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)

        def run(arm):
            if arm == "beauty":
                g.render(w, h, args.beauty_spp, seed=SEED)
                st = g.stats()
            else:
                g.render_aov(w, h, int(arm.split("_")[1]), seed=SEED)
                st = g.aov_stats()
            print(f"{arm}: {st['render_ms']:.1f} ms", file=sys.stderr, flush=True)
            return st

        arms = ["beauty"] + [f"aov_{n}" for n in aov_spp]
        for arm in arms:  # warm-up at the timed shapes
            run(arm)
        rows = {a: [] for a in arms}
        for _ in range(args.reps):
            for arm in arms:
                rows[arm].append(run(arm))
        cov = g.readback_aov()["coverage"]
        result["coverage_mean_last_arm"] = float(cov.mean())
    beauty = min(rows["beauty"], key=lambda s: s["render_ms"])
    beauty_ns = beauty["render_ms"] * 1e6 / beauty["samples"]
    for arm in arms:
        best = min(rows[arm], key=lambda s: s["render_ms"])
        ns = best["render_ms"] * 1e6 / best["samples"]
        row = {"device_ms": best["render_ms"], "device_ms_all": [s["render_ms"] for s in rows[arm]], "ns_per_sample": ns,
               "samples": best["samples"], "extension_rays_per_sample": best["extension_rays"] / best["samples"],
               "launches": best["kernel_launches"], "ns_per_sample_over_beauty": ns / beauty_ns}
        if arm != "beauty":
            paths = min(512 << 20, w * h * int(arm.split("_")[1]))
            row.update({"paths_per_batch": paths, "aov_slot_bytes_per_batch": paths * AOV_BYTES,
                        "batch_bytes": paths * (QUEUE_BYTES + AOV_BYTES)})
        result["arms"][arm] = row
        print(json.dumps({arm: row}), file=sys.stderr, flush=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
