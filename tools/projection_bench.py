#!/usr/bin/env python3
"""projection_bench.py — the cost of each camera projection (rt_gpu_render_projected) per sample.

Scene: BASELINE config 4 (260 192 triangles, 32 emitters, 1000 x 1000 at 250 spp = 1e9 samples), uploaded once, one view
of the scene camera.  Arms, alternating, best of --reps after a warm-up of every arm:
  views       rt_gpu_render_views of the scene camera (the reference point)
  pinhole     rt_gpu_render_projected, RT_PROJ_PINHOLE (the same image, bit for bit; checked)
  thin_lens   aperture 2 % of the scene's extent, focused on the scene's centre
  ortho       half_width = half_height = half the scene's extent
  equirect    the full sphere from the camera position
Per arm: device ms (stats.render_ms), ns per sample, Msamples/s, extension rays per sample and the kernel launches.
Then one profiled pass per arm (rt_gpu_set_profiling: kernels serialised, so slower) gives k_extend's and k_shade's ms
summed over all bounces: depth of field makes the primary rays less coherent, and this is where it would show.  One
JSON line on stdout; the card's name, power limit and max SM clock are part of it.

    python tools/projection_bench.py [--reps 3] [--spp 250]
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

SEED = 7
K_EXTEND, K_SHADE = 1, 2  # rt_stats.kernel_ms slots (rt_gpu.cu KernelKind)


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
    ap.add_argument("--spp", type=int, default=250)
    ap.add_argument("--size", type=int, default=1000)
    args = ap.parse_args()
    import gen_gltf
    import rt_b200
    from rt_b200 import gltf, gpu
    from rt_b200._abi import Projection

    tmp = tempfile.mkdtemp(prefix="rt_projection_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    sc = gltf.load_gltf(gen_gltf.generate("big_lights", tmp), 1.0)
    cam = sc.camera()
    pts = sc.tri_pos.reshape(-1, 3).astype(np.float64)
    lo, hi = pts.min(0), pts.max(0)
    ext = float((hi - lo).max())
    focus = float(np.dot((lo + hi) / 2 - cam.position, cam.forward))
    projs = {"pinhole": Projection.pinhole(), "thin_lens": Projection.thin_lens(0.02 * ext, focus),
             "ortho": Projection.orthographic(ext / 2, ext / 2), "equirect": Projection.equirect()}
    w = h = args.size
    result = {"metric": "ns per sample by camera projection", "card": card(), "scene": "config 4 (big_lights)", "width": w,
              "height": h, "spp": args.spp, "scene_extent": ext, "projections": {k: repr(v) for k, v in projs.items()}, "arms": {}}
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)

        def run(arm):
            if arm == "views":
                g.render_views([cam], w, h, args.spp, seed=SEED)
            else:
                g.render_projected([cam], [projs[arm]], w, h, args.spp, seed=SEED)
            st = g.stats()
            print(f"{arm}: {st['render_ms']:.1f} ms", file=sys.stderr, flush=True)
            return st

        arms = ["views"] + list(projs)
        images = {}
        for arm in arms:  # warm-up at the timed shape; keeps the images of the identity check
            run(arm)
            images[arm] = g.readback()[0][0]
        rows = {a: [] for a in arms}
        for _ in range(args.reps):
            for arm in arms:
                rows[arm].append(run(arm))
        g.set_profiling(True)
        prof = {arm: run(arm) for arm in arms}
        g.set_profiling(False)
        for arm in arms:
            best = min(rows[arm], key=lambda s: s["render_ms"])
            result["arms"][arm] = {
                "device_ms": best["render_ms"], "device_ms_all": [s["render_ms"] for s in rows[arm]],
                "ns_per_sample": best["render_ms"] * 1e6 / best["samples"], "msamples_per_s": best["samples"] / best["render_ms"] * 1e-3,
                "samples": best["samples"], "extension_rays_per_sample": best["extension_rays"] / best["samples"],
                "launches": best["kernel_launches"], "profiled_k_extend_ms": prof[arm]["kernel_ms"][K_EXTEND],
                "profiled_k_shade_ms": prof[arm]["kernel_ms"][K_SHADE]}
            print(json.dumps({arm: result["arms"][arm]}), file=sys.stderr, flush=True)
    result["pinhole_equals_views"] = bool(np.array_equal(images["pinhole"], images["views"]))
    result["pinhole_over_views_device_ms"] = result["arms"]["pinhole"]["device_ms"] / result["arms"]["views"]["device_ms"]
    print(json.dumps(result))


if __name__ == "__main__":
    main()
