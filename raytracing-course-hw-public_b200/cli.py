"""`python -m rt_b200.cli <scene.gltf|scene.txt> <width> <height> <samples> <out.ppm>` — the reference's CLI surface
(src/main.cpp:16-49) for hosts without the reference headers: Python loader (gltf.py, bit-identical flattening),
own BVH build (librt_host), CUDA integrator (librt_gpu), reference tonemap restated in librt_host, binary PPM."""
import os
import sys

from ._abi import Projection


def adaptive_steps(samples):
    """min_samples = step_samples of the CLI's adaptive mode for a maximum of `samples` spp: 16 rounds at most."""
    return max(2, -(-samples // 16))


AOV_NAMES = ("albedo", "normal", "emission", "depth", "coverage")


def parse_aov(text):
    """RT_AOV=<samples> -> samples of the AOV render (unset, empty or 0: off)"""
    if text is None or text == "":
        return 0
    if not text.isdigit():
        raise ValueError(f"RT_AOV={text}: expected the AOV render's samples per pixel, an integer >= 0")
    return int(text)


def aov_paths(out, prefix=""):
    """{name: <stem><prefix>_<name>.pfm} of the AOV buffers written next to the image `out`"""
    stem, _ = os.path.splitext(out)
    return {k: f"{stem}{prefix}_{k}.pfm" for k in AOV_NAMES}


def write_aovs(aovs, out, prefix=""):
    from . import pfm

    for k, path in aov_paths(out, prefix).items():
        pfm.write_pfm(path, aovs[k])


def run_raytracer(scene, width, height, samples, seed=0, n_gpus=1, rel_error=None, projection=None, aov=0):
    """Mirror of run_raytracer(scene, image) (src/raytracer.h:629): float means [H, W, 3] + stats.  With rel_error,
    `samples` is the maximum spp of an adaptive render (rt_gpu_render_adaptive).  With projection (a Projection), the
    scene camera is rendered through it (rt_gpu_render_projected).  With aov > 0 the AOV render (rt_gpu_render_aov) of
    `aov` spp follows on the same camera, projection and seed, and its readback_aov dict is returned third."""
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
            if not aov:
                return mean[0], stats
            rt.render_aov(width, height, aov, seed=seed, cameras=[scene.camera()], projections=[projection], max_paths_in_flight=paths)
            return mean[0], stats, {k: v[0] for k, v in rt.readback_aov().items()}
        if rel_error is None:
            rt.render(width, height, samples, seed=seed, max_paths_in_flight=paths)
        else:
            step = adaptive_steps(samples)
            rt.render_adaptive(width, height, samples, step, step, rel_error, seed=seed, max_paths_in_flight=paths)
        if not aov:
            return rt.readback()
        mean, stats = rt.readback()
        rt.render_aov(width, height, aov, seed=seed, max_paths_in_flight=paths)
        return mean, stats, rt.readback_aov()


def run_views(scene, cameras, width, height, samples, seed=0, n_gpus=1, projections=None, aov=0):
    """Every camera of `cameras` in one rt_gpu_render_views call, or in one rt_gpu_render_projected call when a
    projection of `projections` is not a pinhole: float means [V, H, W, 3] + stats.  With aov > 0 the AOV render of
    `aov` spp over the same views follows, and its readback_aov dict ([V, H, W, ...]) is returned third."""
    from . import gpu

    paths = int(os.environ.get("RT_PATHS", 128 << 20))
    with gpu.RtGpu(n_gpus, 0) as rt:
        rt.upload_scene(scene)
        projected = bool(projections) and any(p != Projection.pinhole() for p in projections)
        if projected:
            rt.render_projected(cameras, projections, width, height, samples, seed=seed, max_paths_in_flight=paths)
        else:
            rt.render_views(cameras, width, height, samples, seed=seed, max_paths_in_flight=paths)
        if not aov:
            return rt.readback()
        mean, stats = rt.readback()
        rt.render_aov(width, height, aov, seed=seed, cameras=cameras, projections=projections if projected else None,
                      max_paths_in_flight=paths)
        return mean, stats, rt.readback_aov()


def parse_frames(text):
    """RT_FRAMES=<count>:<fps> -> (count >= 1, fps > 0)"""
    try:
        count, fps = text.split(":")
        count, fps = int(count), float(fps)
    except ValueError:
        count, fps = 0, 0.0
    if count < 1 or not (0 < fps < float("inf")):
        raise ValueError(f"RT_FRAMES={text}: expected <count>:<fps> with count >= 1 and fps > 0")
    return count, fps


def run_frames(path, width, height, samples, count, fps, out, animation=0, seed=0, n_gpus=1, rel_error=None, projection=None,
               env_map=None):
    """Frames f = 0 .. count - 1 of a glTF animation, frame f at t0 + f / fps: frame 0 is uploaded, every later frame
    moves the uploaded geometry (update_geometry; only the light BVH is built on the host).  Each frame renders its
    camera through `projection` (pinhole by default) with seed + f, at `samples` spp or adaptively with rel_error, to
    <stem>_<f><ext>.  The file's buffers and textures are read once."""
    import time as clock

    from . import gltf, gpu, host

    src = gltf.GltfFile(path)
    t0, _ = gltf.animation_range(src, animation)
    paths = int(os.environ.get("RT_PATHS", 128 << 20))
    proj = projection if projection is not None else Projection.pinhole()
    step = adaptive_steps(samples)
    with gpu.RtGpu(n_gpus, 0) as rt:
        for f, frame_path in enumerate(view_paths(out, count)):
            t = t0 + f / fps
            c0 = clock.perf_counter()
            scene = gltf.load_gltf(src, width / height, build_bvh=f == 0, env_map=env_map, time=t, animation=animation)
            c1 = clock.perf_counter()
            if f == 0:
                rt.upload_scene(scene)
            else:
                rt.update_geometry(gltf.build_light_bvh(scene))
            c2 = clock.perf_counter()
            rt.render_projected([scene.camera()], [proj], width, height, samples, seed=seed + f, max_paths_in_flight=paths,
                                adaptive=None if rel_error is None else (step, step, rel_error))
            mean, stats = rt.readback()
            host.write_ppm(frame_path, host.tonemap_rgb8(mean[0]))
            print(f"rt_gpu frame {f} (t = {t:.6g} s): load {(c1 - c0) * 1e3:.1f} ms, {'upload' if f == 0 else 'update'} "
                  f"{(c2 - c1) * 1e3:.1f} ms, render {stats['render_ms']:.1f} ms", file=sys.stderr)
    return 0


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
        # RT_FRAMES=<count>:<fps> (RT_ANIMATION=<index>, default 0): frames of the glTF's animation, see run_frames
        frames = os.environ.get("RT_FRAMES")
        if textscene.is_text_scene(argv[1]):
            # course text scenes (parity unpinned): width / height / samples of 0 take DIMENSIONS / SAMPLES of the file
            scene = textscene.load_text_scene(argv[1])
            width, height, samples = width or scene.width, height or scene.height, samples or scene.samples
        elif frames is None:
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
        # RT_AOV=<samples>: after the beauty render, the AOV render (rt_gpu_render_aov) of the same camera(s), projection
        # and seed at <samples> spp, written to <stem>_albedo.pfm, _normal, _emission, _depth and _coverage
        try:
            aov = parse_aov(os.environ.get("RT_AOV"))
        except ValueError as e:
            print(e, file=sys.stderr)
            return 1
        if aov and (frames is not None or textscene.is_text_scene(argv[1])):
            print("RT_AOV renders the AOV buffers of one glTF render: it cannot be combined with RT_FRAMES or a text scene",
                  file=sys.stderr)
            return 1
        cameras = os.environ.get("RT_CAMERAS")
        if frames is not None:
            if cameras is not None or textscene.is_text_scene(argv[1]):
                print("RT_FRAMES renders one camera of an animated glTF scene: it cannot be combined with RT_CAMERAS or a "
                      "text scene", file=sys.stderr)
                return 1
            try:
                count, fps = parse_frames(frames)
                animation = int(os.environ.get("RT_ANIMATION", "0"))
                gltf.animation_range(argv[1], animation)
            except ValueError as e:  # also gltf.AnimationError: no animations, or no such animation
                print(f"RT_FRAMES: {e}", file=sys.stderr)
                return 1
            return run_frames(argv[1], width, height, samples, count, fps, argv[5], animation=animation,
                              seed=int(os.environ.get("RT_SEED", "0")), n_gpus=int(os.environ.get("RT_GPUS", "1")),
                              rel_error=rel_error, projection=projection, env_map=os.environ.get("RT_ENV_MAP") or None)
        # RT_CAMERAS=all: every camera node of the glTF in one multi-view render, view i to <stem>_<i><ext>
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
            res = run_views(scene, cams, width, height, samples, seed=int(os.environ.get("RT_SEED", "0")),
                            n_gpus=int(os.environ.get("RT_GPUS", "1")), projections=projs, aov=aov)
            means, stats = res[0], res[1]
            for path, mean in zip(view_paths(argv[5], len(cams)), means):
                host.write_ppm(path, host.tonemap_rgb8(mean))
            if aov:
                for i in range(len(cams)):
                    write_aovs({k: v[i] for k, v in res[2].items()}, argv[5], f"_{i}")
            ms = max(stats["render_ms"], 1e-9)
            print(f"rt_gpu: {len(cams)} views, {ms:.1f} ms, {stats['samples'] / ms * 1e-3:.1f} Msamples/s", file=sys.stderr)
            return 0
        res = run_raytracer(scene, width, height, samples, seed=int(os.environ.get("RT_SEED", "0")),
                            n_gpus=int(os.environ.get("RT_GPUS", "1")), rel_error=rel_error, projection=projection, aov=aov)
        mean, stats = res[0], res[1]
        host.write_ppm(argv[5], host.tonemap_rgb8(mean))
        if aov:
            write_aovs(res[2], argv[5])
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
