#!/usr/bin/env python3
"""update_bench.py — what moving geometry costs: rt_gpu_update_geometry against a re-upload, and what a refit tree costs
the renders that follow.

Scene: BASELINE config 4 (260 192 triangles, 32 emitters).  One JSON line on stdout; the card's name, power limit and max
SM clock are part of it.
  1. Latency, best of --reps with the arms alternating, host clock around each (both calls return after the device
     work): rt_gpu_update_geometry of the scene rotated by 2 degrees (positions, normals and tangents from pageable numpy
     arrays; the light BVH over the new positions is built before the clock starts) and rt_gpu_upload_scene of that
     same scene with no scene BVH (the library builds it on the device).  The first update after an upload also records
     the tree's levels and 4-wide grouping; it is reported on its own.  One more update with RT_TIMING=1 gives the
     serialised phases.
  2. For whole-scene rotations of 0 / 2 / 10 / 45 / 90 degrees about the scene's centre, and for 1 % of the triangles
     (every 100th) moved across the room: the SAH cost of the refit tree and of a tree built for the new positions (both
     downloaded, costed by tests/hostcheck's hc_tree_stats), and a 1000 x 1000 x --spp render of each (device ms, ns per
     sample), then k_extend's ms in a separate profiled pass (kernels serialised).  break_even_msamples: the samples
     after which the extra per-sample time of the refit tree exceeds one re-upload.

    python tools/update_bench.py [--reps 5] [--spp 250]
"""
import argparse
import atexit
import copy
import ctypes as C
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

SEED = 7
K_EXTEND = 1  # rt_stats.kernel_ms slot (rt_gpu.cu KernelKind)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def moved(sc, pos, normals=None):
    from rt_b200 import gltf

    s = copy.copy(sc)
    s.tri_pos = np.ascontiguousarray(pos, np.float32).reshape(sc.n_tris, 3, 3)
    if normals is not None:
        s.tri_normals = np.ascontiguousarray(normals, np.float32).reshape(sc.n_tris, 3, 3)
    return gltf.build_light_bvh(s)


def rotated(sc, deg):
    a = np.radians(deg)
    R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    p = sc.tri_pos.astype(np.float64)
    c = p.reshape(-1, 3).mean(0)
    return moved(sc, (p - c) @ R.T + c, sc.tri_normals.astype(np.float64) @ R.T)


def one_percent_moved(sc):
    """every 100th triangle translated by 60 % of the room's extent along its longest axis (wrapped into the room)"""
    p = sc.tri_pos.astype(np.float64).copy()
    lo, hi = p.reshape(-1, 3).min(0), p.reshape(-1, 3).max(0)
    ax = int(np.argmax(hi - lo))
    sel = np.arange(sc.n_tris) % 100 == 0
    shifted = p[sel][..., ax] + 0.6 * (hi[ax] - lo[ax])
    over = shifted.max(axis=1) > hi[ax]
    shifted[over] -= hi[ax] - lo[ax]
    q = p[sel]
    q[..., ax] = shifted
    p[sel] = q
    return moved(sc, p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--spp", type=int, default=250)
    ap.add_argument("--size", type=int, default=1000)
    args = ap.parse_args()
    import gen_gltf
    from rt_b200 import _abi, gltf, gpu

    hc = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libhostcheck.so"))
    tmp = tempfile.mkdtemp(prefix="rt_update_bench_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)
    A = gltf.load_gltf(gen_gltf.generate("big_lights", tmp), 1.0).without_scene_bvh()
    W = H = args.size
    n_samples = W * H * args.spp
    res = {"bench": "update_bench", "card": card(), "scene": "big_lights (BASELINE config 4)", "n_tris": A.n_tris,
           "width": W, "height": H, "spp": args.spp}

    def tree_cost(rt, sc):
        nodes, objects = rt.debug_bvh(1, _abi.NODE_DTYPE), rt.debug_bvh(2, np.uint32)
        d = sc.desc()
        out = np.zeros(8)
        rc = hc.hc_tree_stats(C.byref(d), nodes.ctypes.data_as(C.c_void_p), C.c_uint64(len(nodes)), objects.ctypes.data_as(C.c_void_p),
                              C.c_uint64(len(objects)), out.ctypes.data_as(C.c_void_p))
        assert rc == 0 and out[5] == 1.0, (rc, out)
        return float(out[6])

    def render(rt):
        rt.render(W, H, args.spp, seed=SEED)
        st = rt.stats()
        rt.set_profiling(True)
        rt.render(W, H, args.spp, seed=SEED)
        k_ext = rt.stats()["kernel_ms"][K_EXTEND]
        rt.set_profiling(False)
        return {"ms": round(st["render_ms"], 2), "ns_per_sample": round(st["render_ms"] * 1e6 / n_samples, 4),
                "extension_rays": st["extension_rays"], "k_extend_ms": round(k_ext, 2)}

    with gpu.RtGpu(1, 0) as rt:
        # 1. latency
        B = rotated(A, 2.0)
        rt.upload_scene(A)
        t = time.perf_counter()
        rt.update_geometry(B)
        first = (time.perf_counter() - t) * 1e3
        upd, upl = [], []
        for _ in range(args.reps):
            rt.upload_scene(A)
            rt.update_geometry(A)  # records the grouping: the timed update below is a steady-state one
            t = time.perf_counter()
            rt.update_geometry(B)
            upd.append((time.perf_counter() - t) * 1e3)
            t = time.perf_counter()
            rt.upload_scene(B)
            upl.append((time.perf_counter() - t) * 1e3)
        rt.upload_scene(A)
        rt.update_geometry(A)
        os.environ["RT_TIMING"] = "1"
        try:
            rt.update_geometry(B)
        finally:
            del os.environ["RT_TIMING"]
        res["latency_ms"] = {"update": round(min(upd), 3), "update_first_after_upload": round(first, 3),
                             "upload": round(min(upl), 3), "update_all": [round(v, 3) for v in upd],
                             "upload_all": [round(v, 3) for v in upl]}
        log = f"update {min(upd):.3f} ms (first after an upload {first:.3f}), upload {min(upl):.3f} ms"
        print(log, file=sys.stderr)
        # 2. refit quality
        rows = []
        for name, make in [(f"rot{d}", (lambda d: lambda s: rotated(s, d))(d)) for d in (0, 2, 10, 45, 90)] + [("move1pct", one_percent_moved)]:
            B = make(A)
            rt.upload_scene(A)
            rt.update_geometry(B)
            refit = {"sah": round(tree_cost(rt, B), 3), **render(rt)}
            rt.upload_scene(B)
            rebuilt = {"sah": round(tree_cost(rt, B), 3), **render(rt)}
            d_ns = refit["ns_per_sample"] - rebuilt["ns_per_sample"]
            row = {"case": name, "refit": refit, "rebuilt": rebuilt,
                   "break_even_msamples": round(min(upl) * 1e6 / d_ns * 1e-6, 1) if d_ns > 0 else None}
            rows.append(row)
            print(json.dumps(row), file=sys.stderr)
        res["refit_quality"] = rows
    print(json.dumps(res))


if __name__ == "__main__":
    main()
