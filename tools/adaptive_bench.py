#!/usr/bin/env python3
"""adaptive_bench.py — what adaptive sampling (rt_gpu_render_adaptive) buys on BASELINE configs 4 and 5.

Per config: an 8192-spp render with another seed is the ground truth; the uniform render (the config's spp, fixed) and
adaptive renders with a maximum of 4x that spp at a few relative-error targets are compared with it.  The targets are
multiples of the uniform render's own RMS relative error (its err map comes from a one-round adaptive render at
min = max = spp, which is that same fixed render).  Per run: device ms (CUDA events of the library, best of --reps),
samples traced, rounds and kernel launches, relMSE (SURVEY.md 8(d)) and 8-bit MAE against the ground truth.  The
headline per config: the fastest adaptive run whose relMSE is at most the uniform render's, and its time against the
uniform one.  Config 5 runs at one GPU's share of an 8-GPU box (3840 x 2160, 512 spp).  One JSON line on stdout;
the card's name and power limit are part of it.

    python tools/adaptive_bench.py [--configs c4,c5] [--reps 2] [--factors 0.5,0.7,1,1.4]
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

CONFIGS = {"c4": (1000, 1000, 1000), "c5": (3840, 2160, 512)}
GT_SPP, GT_SEED, SEED = 8192, 90001, 7


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def rel_mse(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(((a - b) ** 2 / (((a + b) / 2) ** 2 + 1e-4)).mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c4,c5")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--factors", default="0.5,0.7,1,1.4", help="targets as multiples of the uniform render's RMS err")
    args = ap.parse_args()
    import gen_gltf
    import rt_b200  # noqa: F401
    from rt_b200 import gltf, gpu, host

    tmp = tempfile.mkdtemp(prefix="rt_adaptive_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    path = gen_gltf.generate("big_lights", tmp)
    result = {"metric": "adaptive sampling vs uniform spp", "card": card(), "configs": {}}
    with gpu.RtGpu(1, 0) as g:
        for cname in args.configs.split(","):
            w, h, spp = CONFIGS[cname]
            g.upload_scene(gltf.load_gltf(path, w / h))
            g.render(w, h, GT_SPP, seed=GT_SEED)
            truth, _ = g.readback()
            truth8 = host.tonemap_rgb8(truth)

            def measure(fn):
                best = None
                for _ in range(args.reps):
                    fn()
                    st = g.stats()
                    if best is None or st["render_ms"] < best["render_ms"]:
                        best = st
                img, _ = g.readback()
                return best, {"relmse": rel_mse(img, truth),
                              "mae8": float(np.abs(host.tonemap_rgb8(img).astype(np.int32) - truth8.astype(np.int32)).mean())}

            runs = []
            st, q = measure(lambda: g.render(w, h, spp, seed=SEED))
            uniform = {"kind": "uniform", "spp": spp, "ms": st["render_ms"], "samples": st["samples"], "rounds": 1,
                       "launches": st["kernel_launches"], **q}
            runs.append(uniform)
            g.render_adaptive(w, h, spp, spp, 1, 0.0, seed=SEED)  # the same fixed render, with its err map
            _, err = g.readback_adaptive()
            t_rms = float(np.sqrt(np.mean(np.square(err[np.isfinite(err)], dtype=np.float64))))
            max_spp = 4 * spp
            step = max(2, -(-max_spp // 16))
            for f in (float(x) for x in args.factors.split(",")):
                target = f * t_rms
                st, q = measure(lambda: g.render_adaptive(w, h, max_spp, step, step, target, seed=SEED))
                counts, _ = g.readback_adaptive()
                rounds = -(-int(counts.max()) // step)
                runs.append({"kind": "adaptive", "max_spp": max_spp, "min_step": step, "target": target, "target_x_rms": f,
                             "ms": st["render_ms"], "samples": st["samples"], "frac_of_max": st["samples"] / (w * h * max_spp),
                             "rounds_with_work": rounds, "launches": st["kernel_launches"], **q})
            ok = [r for r in runs if r["kind"] == "adaptive" and r["relmse"] <= uniform["relmse"]]
            best = min(ok, key=lambda r: r["ms"]) if ok else None
            result["configs"][cname] = {
                "width": w, "height": h, "spp": spp, "ground_truth_spp": GT_SPP, "uniform_rms_err": t_rms, "runs": runs,
                "headline": {"uniform_ms": uniform["ms"], "adaptive_ms_at_uniform_relmse": best["ms"] if best else None,
                             "speedup": uniform["ms"] / best["ms"] if best else None,
                             "target": best["target"] if best else None}}
            print(json.dumps({cname: result["configs"][cname]["headline"]}), file=sys.stderr, flush=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
