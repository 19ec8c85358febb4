"""`python -m rt_b200.cli <scene.gltf|scene.txt> <width> <height> <samples> <out.ppm>` — the reference's CLI surface
(src/main.cpp:16-49) for hosts without the reference headers: Python loader (gltf.py, bit-identical flattening),
own BVH build (librt_host), CUDA integrator (librt_gpu), reference tonemap restated in librt_host, binary PPM."""
import os
import sys

from ._abi import Projection


def adaptive_steps(samples):
    """min_samples = step_samples of the CLI's adaptive mode for a maximum of `samples` spp: 16 rounds at most."""
    return max(2, -(-samples // 16))


def run_raytracer(scene, width, height, samples, seed=0, n_gpus=1, rel_error=None, projection=None):
    """Mirror of run_raytracer(scene, image) (src/raytracer.h:629): float means [H, W, 3] + stats.  With rel_error,
    `samples` is the maximum spp of an adaptive render (rt_gpu_render_adaptive).  With projection (a Projection), the
    scene camera is rendered through it (rt_gpu_render_projected)."""
    from . import gpu, textscene

    with gpu.RtGpu(n_gpus, 0) as rt:
        if isinstance(scene, textscene.TextScene):
            rt.upload_text_scene(scene)
        else:
            rt.upload_scene(scene)
        # one-shot command: 128 Mi paths per batch (17 GB of queues instead of 68 GB), see host/main_ref_host.cpp
        paths = int(os.environ.get("RT_PATHS", 128 << 20))
        if projection is not None:
            step = adaptive_steps(samples)
            rt.render_projected([scene.camera()], [projection], width, height, samples, seed=seed, max_paths_in_flight=paths,
                                adaptive=None if rel_error is None else (step, step, rel_error))
            mean, stats = rt.readback()
            return mean[0], stats
        if rel_error is None:
            rt.render(width, height, samples, seed=seed, max_paths_in_flight=paths)
        else:
            step = adaptive_steps(samples)
            rt.render_adaptive(width, height, samples, step, step, rel_error, seed=seed, max_paths_in_flight=paths)
        return rt.readback()


def run_views(scene, cameras, width, height, samples, seed=0, n_gpus=1, projections=None):
    """Every camera of `cameras` in one rt_gpu_render_views call, or in one rt_gpu_render_projected call when a
    projection of `projections` is not a pinhole: float means [V, H, W, 3] + stats."""
    from . import gpu

    paths = int(os.environ.get("RT_PATHS", 128 << 20))
    with gpu.RtGpu(n_gpus, 0) as rt:
        rt.upload_scene(scene)
        if projections and any(p != Projection.pinhole() for p in projections):
            rt.render_projected(cameras, projections, width, height, samples, seed=seed, max_paths_in_flight=paths)
        else:
            rt.render_views(cameras, width, height, samples, seed=seed, max_paths_in_flight=paths)
        return rt.readback()


def view_paths(out, n):
    """<stem>_<i><ext> for the n views of RT_CAMERAS=all"""
    stem, ext = os.path.splitext(out)
    return [f"{stem}_{i}{ext}" for i in range(n)]


def main(argv=None):
    argv = sys.argv if argv is None else argv
    if len(argv) < 6:
        print(f"Too few arguments: expected 6, got {len(argv) - 1}", file=sys.stderr)
        return 1
    from . import gltf, host, textscene

    try:
        width, height, samples = int(argv[2]), int(argv[3]), int(argv[4])
        if textscene.is_text_scene(argv[1]):
            # course text scenes (parity unpinned): width / height / samples of 0 take DIMENSIONS / SAMPLES of the file
            scene = textscene.load_text_scene(argv[1])
            width, height, samples = width or scene.width, height or scene.height, samples or scene.samples
        else:
            scene = gltf.load_gltf(argv[1], width / height, env_map=os.environ.get("RT_ENV_MAP") or None)
        # RT_ADAPTIVE=<rel_error>: `samples` is the maximum spp; every pixel stops once its relative error is reached
        adaptive = os.environ.get("RT_ADAPTIVE")
        rel_error = float(adaptive) if adaptive else None
        # RT_PROJECTION=thin_lens:<aperture>:<focus> | ortho:<half_w>:<half_h> | equirect | pinhole: the projection of
        # the rendered camera(s); with RT_CAMERAS=all, each camera node otherwise keeps the glTF's own projection
        projection = os.environ.get("RT_PROJECTION")
        if projection:
            if textscene.is_text_scene(argv[1]):
                print("RT_PROJECTION applies to glTF scenes only", file=sys.stderr)
                return 1
            try:
                projection = Projection.parse(projection)
            except ValueError as e:
                print(f"RT_PROJECTION: {e}", file=sys.stderr)
                return 1
        else:
            projection = None
        # RT_CAMERAS=all: every camera node of the glTF in one multi-view render, view i to <stem>_<i><ext>
        cameras = os.environ.get("RT_CAMERAS")
        if cameras is not None:
            if cameras != "all":
                print(f"RT_CAMERAS={cameras}: the only value is 'all'", file=sys.stderr)
                return 1
            if rel_error is not None or textscene.is_text_scene(argv[1]):
                print("RT_CAMERAS=all renders glTF scenes at a fixed spp: it cannot be combined with RT_ADAPTIVE or a "
                      "text scene", file=sys.stderr)
                return 1
            cams = scene.cameras or [scene.camera()]  # no camera node: the scene's default camera
            projs = [projection] * len(cams) if projection is not None else scene.projections or [Projection.pinhole()]
            means, stats = run_views(scene, cams, width, height, samples, seed=int(os.environ.get("RT_SEED", "0")),
                                     n_gpus=int(os.environ.get("RT_GPUS", "1")), projections=projs)
            for path, mean in zip(view_paths(argv[5], len(cams)), means):
                host.write_ppm(path, host.tonemap_rgb8(mean))
            ms = max(stats["render_ms"], 1e-9)
            print(f"rt_gpu: {len(cams)} views, {ms:.1f} ms, {stats['samples'] / ms * 1e-3:.1f} Msamples/s", file=sys.stderr)
            return 0
        mean, stats = run_raytracer(scene, width, height, samples, seed=int(os.environ.get("RT_SEED", "0")),
                                    n_gpus=int(os.environ.get("RT_GPUS", "1")), rel_error=rel_error, projection=projection)
        host.write_ppm(argv[5], host.tonemap_rgb8(mean))
        ms = max(stats["render_ms"], 1e-9)
        print(f"rt_gpu: {ms:.1f} ms, {stats['samples'] / ms * 1e-3:.1f} Msamples/s", file=sys.stderr)
        if rel_error is not None:
            full = width * height * samples
            print(f"rt_gpu adaptive (rel_error {rel_error:g}): {stats['samples']} samples traced, "
                  f"{stats['samples'] / full:.3f} of {full}", file=sys.stderr)
    except RuntimeError as e:
        print(e, file=sys.stderr)
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
