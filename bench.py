#!/usr/bin/env python3
"""bench.py — Msamples/s of the path-tracing hot path on B200 (BASELINE.json metric).

Workload (config 4 of BASELINE.json): the synthetic "Sponza-scale" glTF of SURVEY.md 8(d) — 260 192 triangles,
textured, 32 emissive triangles — at 1000 x 1000 pixels, 1000 spp.  One step = one full render of that image
(1e9 pixel-samples).  With N GPUs (one process per GPU, torchrun) the FIXED 1000 spp are split: rank r renders
samples [1000 r / N, 1000 (r+1) / N) of every pixel ("strong" scaling — the north star's "1000x1000, 1000 spp on
8 x B200", the GPU analogue of the reference's span pool, raytracer.h:635-665), followed by the path's single
collective: one NCCL reduce(sum) of the W*H*4 float accumulation buffer to rank 0, inside the timed region.
`--scaling weak` renders 1000 spp PER GPU instead (a 1000 N spp image); `--config c5` is BASELINE config 5
(3840 x 2160, 4096 spp split over the ranks).  After the timed region an N > 1 run CHECKS its reduced image against
a single-GPU render of the same sample set on rank 0 (`parity_check`).

  value        device-timed (CUDA events) samples/s of K steps, scene resident in HBM
  e2e          the same through the public C ABI with (pinned) host buffers every step: rt_gpu_upload_scene (H2D of
               the scene's arrays, BVH build + re-packing on the device) -> rt_gpu_render -> rt_gpu_readback (D2H of
               the float means)
  roofline     dominant kernel k_extend (BVH traversal) against the measured FP32 FMA rate; algorithmic
               flops = 24/box test + 70/triangle test of the REFERENCE's traversal (SURVEY.md 8(d)), counted by
               the oracle on a sample of the same workload
  cpu_baseline the unmodified reference (oracle/_ref, kind "reference") or the oracle port, timed on this box's
               host cores on a bounded sample of the same scene

`--impl reference` times the reference's own CPU implementation instead (same metric / config keys).
`--dump-outputs DIR` writes the per-pixel sums of the last timed step to DIR (fixed seed and scene: two builds run with
the same arguments can be compared output for output).
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scenes")]

SCENE = "big_lights"
WIDTH = HEIGHT = 1000
SPP = 1000
METRIC = "Msamples/s"
FLOP_BOX, FLOP_TRI = 24.0, 70.0  # SURVEY.md 8(d): slab test, Cramer triangle test


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to
# stdout), so file descriptor 1 is pointed at stderr for the whole run and the result line goes to a
# private duplicate of the original stdout.
_RESULT_FD = None


def _capture_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


_SCENE_DIR = None


def scene_path(name):
    """Deterministic synthetic scene, generated on first use into a temporary directory of this process (the tree
    may be read-only; one private copy per rank: no write races), removed at exit."""
    global _SCENE_DIR
    import gen_gltf

    if _SCENE_DIR is None:
        _SCENE_DIR = tempfile.mkdtemp(prefix="rt_b200_scenes_")
        atexit.register(shutil.rmtree, _SCENE_DIR, ignore_errors=True)
    p = os.path.join(_SCENE_DIR, name + ".gltf")
    if not os.path.exists(p):
        gen_gltf.generate(name, _SCENE_DIR)
    return p


DUMP_BYTES = 64 * 10**6  # all files of the dump, .npy headers included
NPY_HEADER_MAX = 4096  # room left per file for its .npy header (128 bytes in practice)
DUMP_SEED = 20261020


def dump_outputs(out_dir, sums, w, h):
    """The per-pixel float sums the timed path returned (W*H*4 float32: rgb + unused w) as accum_sums.npy [H, W, 4].
    Above DUMP_BYTES a fixed, seeded sample of the pixels is written instead: accum_sums.npy [k, 4] and the row-major
    pixel index of each row in accum_pixel_index.npy."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    sums = np.ascontiguousarray(sums, np.float32).reshape(h, w, 4)
    if sums.nbytes + NPY_HEADER_MAX <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "accum_sums.npy"), sums)
        log(f"dump-outputs: accum_sums.npy {sums.shape} -> {out_dir}")
        return
    k = (DUMP_BYTES - 2 * NPY_HEADER_MAX) // (sums.itemsize * 4 + 8)  # + one float64 pixel index per row
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(w * h, size=k, replace=False))
    np.save(os.path.join(out_dir, "accum_sums.npy"), sums.reshape(-1, 4)[idx])
    np.save(os.path.join(out_dir, "accum_pixel_index.npy"), idx.astype(np.float64))
    log(f"dump-outputs: {k} of {w * h} pixels (seed {DUMP_SEED}) -> {out_dir}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_throughput(budget_s, width=500, height=500):
    """Msamples/s of the reference CPU path on `SCENE`: wall(run_raytracer, spp_hi) - wall(spp = 1), which
    cancels the two BVH builds inside run_raytracer (raytracer.h:633); all hardware threads
    (raytracer.h:636).  Falls back to the oracle port when oracle/_ref was not built."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_lib as O

    cores = os.cpu_count() or 1
    gltf = scene_path(SCENE)
    if O.have_ref_tool():
        def wall(spp):
            r = subprocess.run([O.REF_TOOL, "time", gltf, str(width), str(height), str(spp)], capture_output=True,
                               text=True, check=True)
            return float(r.stderr.strip().splitlines()[-1])

        t1 = wall(1)
        t5 = wall(5)
        rate = width * height * 4 / max(t5 - t1, 1e-3)  # samples/s pilot
        spp_hi = int(max(8, min(4096, 1 + budget_s * rate / (width * height))))
        thi = wall(spp_hi)
        v = width * height * (spp_hi - 1) / max(thi - t1, 1e-6) / 1e6
        return {"value": v, "unit": METRIC, "cores": cores, "kind": "reference",
                "sample": f"{SCENE} {width}x{height}, run_raytracer wall(spp={spp_hi}) - wall(spp=1) = "
                          f"{thi - t1:.2f} s, unmodified reference (oracle/_ref/ref_tool time)"}
    import rt_b200
    from rt_b200 import gltf as gl

    scene = gl.load_gltf(gltf, width / height)
    t0 = time.perf_counter()
    O.render(scene, width, height, 1, rng_mode=O.RNG_MINSTD, n_threads=cores)
    rate = width * height / (time.perf_counter() - t0)
    spp = int(max(2, min(4096, budget_s * rate / (width * height))))
    t0 = time.perf_counter()
    O.render(scene, width, height, spp, rng_mode=O.RNG_MINSTD, n_threads=cores)
    dt = time.perf_counter() - t0
    return {"value": width * height * spp / dt / 1e6, "unit": METRIC, "cores": cores, "kind": "port",
            "sample": f"{SCENE} {width}x{height} x {spp} spp in {dt:.2f} s, oracle/pt_oracle.c (minstd mode)"}


def reference_counts():
    """Per-extension-ray work of the REFERENCE's traversal on this workload (oracle counters)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_lib as O
    from rt_b200 import gltf as gl

    scene = gl.load_gltf(scene_path(SCENE), WIDTH / HEIGHT)
    _, st = O.render(scene, 100, 100, 4, rng_mode=O.RNG_PHILOX, seed=1)
    e = max(st["extension_rays"], 1)
    return {"box_tests_per_ray": st["box_tests"] / e, "tri_tests_per_ray": st["tri_tests"] / e,
            "nodes_per_ray": st["nodes_visited"] / e, "rays_per_sample": e / st["samples"],
            "light_box_per_lray": st["light_box_tests"] / max(st["light_pdf_rays"], 1),
            "light_tri_per_lray": st["light_tri_tests"] / max(st["light_pdf_rays"], 1)}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    world = args.gpus
    spp_total = args.spp * world if args.scaling == "weak" else args.spp
    # each step is a bounded sample sized so that the whole run ends within a few minutes
    per_step = max(2.0, min(20.0, 150.0 / max(steps + warm, 1)))
    vals = []
    for i in range(warm + steps):
        r = cpu_throughput(per_step, 250, 250)
        if i >= warm:
            vals.append(r)
    v = sum(x["value"] for x in vals) / len(vals)
    samples_per_step = args.width * args.height * spp_total
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": METRIC, "n_gpus": args.gpus, "steps": steps,
           "warmup": warm, "ms_per_step": samples_per_step / (v * 1e6) * 1e3, "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": v / 0.355, "dtype": "f32", "data": "synthetic",
           "config": config_dict(args, world),
           "note": "CPU arm: each step is a bounded sample (250x250) of the workload; ms_per_step is the "
                   "extrapolated full step",
           "cpu_baseline": {**vals[-1], "value": v},
           "e2e": {"value": v, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


def config_dict(args, n_gpus):
    """The workload both arms are quoted on (identical keys and values for --impl b200 and --impl reference)."""
    w, h = args.width, args.height
    spp_total = args.spp * n_gpus if args.scaling == "weak" else args.spp
    if (w, h, spp_total) == (WIDTH, HEIGHT, SPP):
        name = "BASELINE config 4"
    elif (w, h, spp_total) == (3840, 2160, 4096):
        name = "BASELINE config 5"
    else:
        name = "BASELINE config 4 scene at a non-default size"
    return {"workload": f"{name}: synthetic Sponza-scale glTF '{args.scene}' (260192 triangles, textured, 32 emissive), "
                        f"{w}x{h}, {spp_total} spp, ray depth 8",
            "scene": args.scene, "width": w, "height": h, "spp_total": spp_total, "spp_per_gpu": spp_total / n_gpus,
            "parallelism": f"sample-split x{n_gpus} + 1 NCCL reduce" if n_gpus > 1 else "single GPU",
            "l2": "256 MiB written between steps; per-step path-queue traffic (>100 GB) far exceeds the 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def run_gpu_arm(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    import rt_b200  # noqa: F401
    from rt_b200 import dist as rtdist
    from rt_b200 import gltf as gl
    from rt_b200 import gpu

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (this backend has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    w, h = args.width, args.height
    spp_total = args.spp * world if args.scaling == "weak" else args.spp
    t0 = time.perf_counter()
    scene = gl.load_gltf(scene_path(args.scene), w / h)
    t_load = time.perf_counter() - t0
    rt = gpu.RtGpu(1, local_rank)
    t0 = time.perf_counter()
    rt.upload_scene(scene)
    t_upload = time.perf_counter() - t0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    seed = 20261018

    def step(i):
        flush.fill_(i & 255)  # L2 flush between iterations
        sums = rtdist.render_distributed(rt, w, h, spp_total, seed, rank, world, local_rank, args.paths)
        return sums

    for i in range(args.warmup):
        step(i)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    rays = [0, 0]
    e0.record()
    for i in range(args.steps):
        sums = step(i)
        st = rt.stats()
        launches += st["kernel_launches"] + (1 if world > 1 else 0)
        rays[0] += st["extension_rays"]
        rays[1] += st["light_pdf_rays"]
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    ray_t = torch.tensor(rays, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(ray_t, op=dist.ReduceOp.SUM)
    clk = clocks.stop() if rank == 0 else None
    total_ms = float(ms.item())
    samples_all = float(w) * h * spp_total * args.steps
    value = samples_all / (total_ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:  # the reduced sums of the last timed step, before anything renders again
        dump_outputs(args.dump_outputs, sums.cpu().numpy(), w, h)

    # the N-rank image of the last timed step, for the parity check below
    img_n = rt.readback()[0] if (rank == 0 and world > 1) else None

    # ---- e2e: host buffers every step through the C ABI ------------------------------------------------
    host_out = torch.empty((h, w, 3), dtype=torch.float32, pin_memory=True).numpy()  # pinned: the D2H lands directly
    # The step's input is the scene as a host passes it: per-triangle arrays, materials, textures and the light BVH — no
    # scene BVH (rt_gpu.h: the library builds it, on the device) — held in PINNED host memory.
    e2e_scene = scene.without_scene_bvh()
    e2e_scene._normalise()

    def pinned(a):
        a = np.ascontiguousarray(a)
        t = torch.from_numpy(a.view(np.uint8).reshape(-1)).pin_memory()
        return t.numpy().view(a.dtype).reshape(a.shape)

    for name in ("tri_pos", "tri_normals", "tri_uv", "tri_tangents", "tri_material", "texels"):
        if getattr(e2e_scene, name) is not None and getattr(e2e_scene, name).size:
            setattr(e2e_scene, name, pinned(getattr(e2e_scene, name)))
    scene_bytes = sum(a.nbytes for a in e2e_scene._sections() if a is not None)

    def e2e_step():
        rt.upload_scene(e2e_scene)  # H2D of the host's arrays + BVH build, re-packing and quantisation on the device
        sums = rtdist.render_distributed(rt, w, h, spp_total, seed, rank, world, local_rank, args.paths)
        if rank == 0:
            rt.readback_into(host_out)  # D2H of the per-pixel sums, / spp on the host
        return sums

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = samples_all / float(e2e_s.item()) / 1e6

    # ---- parity of the multi-GPU result (N > 1): the reduced image == one GPU rendering the same samples ------
    # (reference semantics: the union of the spans, raytracer.h:639-659; Philox is keyed by the global sample index,
    # so only the float summation order differs).  Two checks: the benchmark's own image (full spp, unless that
    # would take more than a few seconds on one GPU), and a 16-spp image at the multi-GPU test's tolerance.
    parity = None
    if world > 1:
        chk_spp = max(16, 2 * world)
        rtdist.render_distributed(rt, w, h, chk_spp, seed, rank, world, local_rank, args.paths)
        small_n = rt.readback()[0] if rank == 0 else None
        barrier()
        if rank == 0:
            def cmp(a, b, rtol, atol):
                fin = np.isfinite(b)
                rel = np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1e-6)
                return {"max_rel": float(rel.max()) if rel.size else 0.0, "rtol": rtol, "atol": atol,
                        "allclose": bool(np.allclose(a, b, rtol=rtol, atol=atol))}

            rt.render(w, h, chk_spp, seed=seed, max_paths_in_flight=args.paths)
            parity = {"n_ranks": world, "small": {"spp": chk_spp, **cmp(small_n, rt.readback()[0], 2e-6, 1e-7)}}
            if float(w) * h * spp_total <= 2.5e9:
                rt.render(w, h, spp_total, seed=seed, max_paths_in_flight=args.paths)
                # sequential float sums of up to 512 samples per batch: reordering moves a pixel by ~1e-6 relative
                parity["bench_image"] = {"spp": spp_total, **cmp(img_n, rt.readback()[0], 2e-5, 1e-6)}
            parity["max_rel"] = max(v["max_rel"] for v in parity.values() if isinstance(v, dict))
            parity["ok"] = all(v["allclose"] for v in parity.values() if isinstance(v, dict))
            log("parity_check", parity)
        barrier()

    # ---- roofline of the dominant kernel + CPU baseline (rank 0 only) ---------------------------------
    roof = cpu = counts = None
    kernel_ms = None
    if rank == 0:
        rt.set_profiling(True)
        sb, se = rtdist.sample_range(spp_total, rank, world)
        rt.render(w, h, spp_total, seed=seed, sample_begin=sb, sample_end=se, max_paths_in_flight=args.paths)
        pst = rt.stats()
        rt.set_profiling(False)
        kernel_ms = {"generate": pst["kernel_ms"][0], "extend": pst["kernel_ms"][1], "shade": pst["kernel_ms"][2],
                     "accumulate": pst["kernel_ms"][3], "lightpdf": pst["kernel_ms"][5], "render_total": pst["render_ms"]}
        peak = rt.fp32_peak_tflops()
        counts = reference_counts()
        flop_per_ray = FLOP_BOX * counts["box_tests_per_ray"] + FLOP_TRI * counts["tri_tests_per_ray"]
        # launches of a batch: k_generate, depth x (k_extend + k_shade), k_accumulate and, with lights, k_lightpdf_list for
        # every queue but the camera rays'
        has_lights = len(scene.light_bvh.objects) > 0
        per_batch = 2 + 2 * scene.ray_depth + (max(scene.ray_depth - 1, 0) if has_lights else 0)
        n_ext_launches = max(1, (pst["kernel_launches"] // per_batch) * scene.ray_depth)
        achieved = flop_per_ray * pst["extension_rays"] / (pst["kernel_ms"][1] * 1e-3) / 1e12
        # the light-pdf traversals were a mode of k_extend until round 2 (no algorithmic flop credited, their time in
        # the denominator); they now run in k_lightpdf_list: the figure with its time added back, for comparison
        ext_plus_light_ms = pst["kernel_ms"][1] + pst["kernel_ms"][5]
        traffic = traffic_note = None
        try:  # DRAM bytes per extension ray of k_extend from the committed `ncu --set full` capture
            with open(os.path.join(ROOT, "profiles", "k_extend_dram.json")) as f:
                tj = json.load(f)
            traffic = tj["dram_bytes_per_ray"] * pst["extension_rays"] / n_ext_launches
            traffic_note = tj["note"]
        except (OSError, KeyError, ValueError):
            pass
        roof = {"bound": "fp32", "kernel": "k_extend", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": "measured on this GPU by rt_gpu_fp32_peak (FFMA loop); MEASURED_PEAKS.json has no FP32 "
                               "entry; nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4",
                "algorithmic_flop_per_ray": flop_per_ray, "rays_per_launch": pst["extension_rays"] / n_ext_launches,
                "avg_launch_ms": pst["kernel_ms"][1] / n_ext_launches, "launches": n_ext_launches,
                "extend_share_of_step": pst["kernel_ms"][1] / max(pst["render_ms"], 1e-9),
                "mrays_per_s_in_kernel": pst["extension_rays"] / (pst["kernel_ms"][1] * 1e-3) / 1e6,
                "frac_with_lightpdf_kernel_time": (flop_per_ray * pst["extension_rays"] / (ext_plus_light_ms * 1e-3) / 1e12 / peak) if peak else None}
        if world == 1:
            cpu = cpu_throughput(args.cpu_budget)

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
               "scaling": args.scaling, "vs_baseline": value / 0.355, "dtype": "f32", "data": "synthetic",
               "config": config_dict(args, world),
               "mrays_per_s": {"extension": float(ray_t[0].item()) / (total_ms * 1e-3) / 1e6,
                               "light_pdf": float(ray_t[1].item()) / (total_ms * 1e-3) / 1e6},
               "e2e": {"value": e2e_value, "unit": METRIC, "h2d_bytes_per_step": int(scene_bytes),
                       "d2h_bytes_per_step": int(w * h * 12)},
               "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
               "parity_check": parity,
               "kernel_ms_profiled_step": kernel_ms, "reference_work_per_ray": counts,
               "host_s": {"load_and_bvh_build": t_load, "first_upload": t_upload},
               "vs_baseline_note": "0.355 Msamples/s = README.md:4 (Sponza 1000x1000x1000spp in ~47 min, unknown CPU)"}
        emit(out)
    barrier()
    rt.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default=SCENE)
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--height", type=int, default=HEIGHT)
    ap.add_argument("--spp", type=int, default=None,
                    help="samples per pixel of the image (strong scaling: split over the GPUs; weak: per GPU)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--config", default="c4", choices=["c4", "c5"], help="BASELINE config 4 (default) or 5")
    ap.add_argument("--paths", type=int, default=0, help="paths in flight per batch (0 = library default)")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the per-pixel sums of the last timed step to DIR/*.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the GPU path (--impl b200)")
    if args.config == "c5":
        args.width, args.height = 3840, 2160
    if args.spp is None:
        args.spp = 4096 // (args.gpus if args.scaling == "weak" else 1) if args.config == "c5" else SPP
    _capture_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    libs = [os.path.join(ROOT, "raytracing-course-hw-public_b200", n) for n in ("librt_gpu.so", "librt_host.so")]
    libs.append(os.path.join(ROOT, "oracle", "libpt_oracle.so"))
    if not all(os.path.exists(p) for p in libs):
        if rank == 0:
            import __graft_entry__ as entry

            entry.build()
        else:
            while not all(os.path.exists(p) for p in libs):
                time.sleep(0.5)
            time.sleep(2.0)
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    run_gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
