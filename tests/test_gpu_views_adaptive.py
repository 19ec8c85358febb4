"""Adaptive multi-view rendering (rt_gpu_render_views_adaptive) on the GPU.  The call is rt_gpu_render_adaptive over the
stacked image of rt_gpu_render_views: pixel p of view v is keyed (view_base + v) * W * H + p and every pixel receives
the sample prefix [0, n_p).  So one view of the scene camera is rt_gpu_render_adaptive, view v of a call is a one-view
call with view_base = v, and a pixel with count n is rt_gpu_render_views of samples [0, n): the tests check all three
bit for bit, with sizes at which every round of every compared call is one batch, plus the stopping rule, the moments,
pixel ranges, every error status, the launch bound and two devices."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN
from views_scene import yawed

import rt_b200
from rt_b200 import _abi, gpu

pytestmark = pytest.mark.gpu

W, H = 96, 64  # whole 8 x 4 tiles: one tile never crosses a view


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


def fan(scene, n, spread=20.0):
    """n cameras: the scene camera yawed evenly over +-spread degrees"""
    own = scene.camera()
    return [yawed(own, a) for a in np.linspace(-spread, spread, n)]


def _median_target(rt, cams, w, h, seed):
    """The stopping target taken from the data: the median err after one 4-sample round, over the pixels with noise
    (the constant sky has err 0, and a target of 0 never stops a pixel)."""
    rt.render_views_adaptive(cams, w, h, 4, 4, 4, 0.0, seed=seed)
    err = rt.readback_adaptive()[1]
    return float(np.median(err[err > 0]))


@pytest.mark.parametrize("name", ["tiny", "small_lights", "tiny_env", "texmaps"])
def test_one_view_of_the_scene_camera_is_render_adaptive(name, rt, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    rt.upload_scene(sc)
    seed, lo, step, hi = 31, 4, 4, 24
    target = _median_target(rt, [sc.camera()], w, h, seed)
    rt.render_adaptive(w, h, hi, lo, step, target, seed=seed)
    ref, st = rt.readback()
    ref8 = rt.readback_rgb8()
    ref_c, ref_e = rt.readback_adaptive()
    assert len(np.unique(ref_c)) >= 2  # the target stops some pixels early
    rt.render_views_adaptive([sc.camera()], w, h, hi, lo, step, target, seed=seed)
    img, st_v = rt.readback()
    counts, err = rt.readback_adaptive()
    assert img.shape == (1, h, w, 3) and counts.shape == (1, h, w) and err.shape == (1, h, w)
    assert np.array_equal(img[0], ref) and np.array_equal(rt.readback_rgb8()[0], ref8)
    assert np.array_equal(counts[0], ref_c) and np.array_equal(err[0], ref_e)
    assert st_v["samples"] == st["samples"] == int(ref_c.sum())
    assert st_v["kernel_launches"] == st["kernel_launches"]


def test_views_equal_one_view_calls(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 5)
    seed, lo, step, hi = 3, 4, 4, 24
    target = _median_target(rt, cams, W, H, seed)
    rt.render_views_adaptive(cams, W, H, hi, lo, step, target, seed=seed)
    many, st = rt.readback()
    many_c, many_e = rt.readback_adaptive()
    assert many.shape == (5, H, W, 3) and st["samples"] == int(many_c.sum())
    assert len(np.unique(many_c)) >= 3
    for v, cam in enumerate(cams):
        rt.render_views_adaptive([cam], W, H, hi, lo, step, target, seed=seed, view_base=v)
        one = rt.readback()[0][0]
        c, e = rt.readback_adaptive()
        assert np.array_equal(many[v], one) and np.array_equal(many_c[v], c[0]) and np.array_equal(many_e[v], e[0]), v
    # view_base = b: the views of the view_base = 0 call from b on
    b = 2
    rt.render_views_adaptive(cams[b:], W, H, hi, lo, step, target, seed=seed, view_base=b)
    shifted, _ = rt.readback()
    c, e = rt.readback_adaptive()
    assert np.array_equal(shifted, many[b:]) and np.array_equal(c, many_c[b:]) and np.array_equal(e, many_e[b:])


def _views_in_steps(rt, cams, n, seed, first, step):
    """samples [0, first), [first, first + step) ... [.., n) of render_views accumulated into one n-spp image"""
    rt.render_views(cams, W, H, n, seed=seed, sample_begin=0, sample_end=min(first, n))
    s = first
    while s < n:
        rt.render_views(cams, W, H, n, seed=seed, sample_begin=s, sample_end=min(s + step, n), accumulate=True)
        s += step
    return rt.readback()[0]


def test_adaptive_views_equal_truncated_render_views(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    seed, lo, step, hi = 5, 4, 4, 24
    target = _median_target(rt, cams, W, H, seed)
    rt.render_views_adaptive(cams, W, H, hi, lo, step, target, seed=seed)
    img, st = rt.readback()
    counts, err = rt.readback_adaptive()
    values = sorted(set(counts.ravel().tolist()))
    print(f"target {target:.4f}: counts {values}, {counts.sum() / (3 * W * H * hi):.3f} of the maximum traced")
    assert len(values) >= 3 and lo in values and hi in values
    assert all((v - lo) % step == 0 for v in values) and st["samples"] == int(counts.sum())
    # the stopping invariant: n = max, or err <= target now and > target one round earlier (the err map of a target-0
    # render to n - step, which sums the same sample ranges)
    assert np.all(err[counts < hi] <= target)
    assert np.all(counts[err > target] == hi)
    for n in values:
        sel = counts == n
        if lo < n:
            rt.render_views_adaptive(cams, W, H, n - step, lo, step, 0.0, seed=seed)
            prev_c, prev_e = rt.readback_adaptive()
            assert np.all(prev_c == n - step)
            assert not np.any(prev_e[sel] <= target), n  # (NaN, an infinite sample, never stops)
        # bit identity with render_views of samples [0, n) in the rounds' sample ranges
        fixed = _views_in_steps(rt, cams, n, seed, lo, step)
        assert np.array_equal(img[sel], fixed[sel]), n


def test_target_zero_with_min_equal_max_is_render_views(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    rt.render_views(cams, W, H, 6, seed=9)
    fixed, st = rt.readback()
    fixed8 = rt.readback_rgb8()
    rt.render_views_adaptive(cams, W, H, 6, 6, 1, 0.0, seed=9)
    img, st2 = rt.readback()
    counts, _ = rt.readback_adaptive()
    assert np.array_equal(img, fixed) and np.all(counts == 6)
    assert np.array_equal(rt.readback_rgb8(), fixed8)
    assert st2["samples"] == st["samples"] == 3 * W * H * 6


def test_error_map_matches_host_moments(rt, golden_scene):
    """min = max = 8 at target 0: every pixel of every view has 8 samples; its err against float64 moments of 8
    one-sample render_views calls (test_gpu_adaptive's tolerance)."""
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    seed, n, floor = 13, 8, 1e-3
    ys = []
    for s in range(n):
        rt.render_views(cams, W, H, 1, seed=seed, sample_begin=s, sample_end=s + 1)
        ys.append(rt.readback()[0].astype(np.float64).sum(axis=3) / 3.0)
    y = np.stack(ys)
    S, Q = y.sum(axis=0), (y * y).sum(axis=0)
    m = S / n
    var = np.maximum(Q / n - m * m, 0.0) * n / (n - 1)
    want = np.sqrt(var / n) / (m + floor)
    rt.render_views_adaptive(cams, W, H, n, n, 1, 0.0, abs_floor=floor, seed=seed)
    counts, err = rt.readback_adaptive()
    assert np.all(counts == n)
    atol = np.sqrt(16 * 2.0 ** -23 * (Q / n) / n) / (m + floor)
    ok = np.abs(err - want) <= 1e-4 * want + atol
    print(f"err: {ok.mean() * 100:.3f} % within tolerance, max |diff| {np.abs(err - want).max():.3g}")
    assert ok.all()


def test_pixel_range_across_views(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 4)
    seed, lo, step, hi = 12, 4, 4, 16
    target = _median_target(rt, cams, W, H, seed)
    rt.render_views_adaptive(cams, W, H, hi, lo, step, target, seed=seed)
    full, _ = rt.readback()
    full_c, full_e = rt.readback_adaptive()
    rgb8 = rt.readback_rgb8()
    ptr, nf = rt.accum_device_ptr()
    assert rgb8.shape == (4, H, W, 3) and ptr and nf == 4 * W * H * 4
    b, e = W * H - 100, 2 * W * H + 37  # from view 0 through view 1 into view 2
    rt.render_views_adaptive(cams, W, H, hi, lo, step, target, seed=seed, pixel_begin=b, pixel_end=e)
    part, st = rt.readback()
    c, er = rt.readback_adaptive()
    flat, flat_full = part.reshape(-1, 3), full.reshape(-1, 3)
    c, er, fc, fe = c.ravel(), er.ravel(), full_c.ravel(), full_e.ravel()
    assert np.array_equal(flat[b:e], flat_full[b:e]) and np.array_equal(c[b:e], fc[b:e]) and np.array_equal(er[b:e], fe[b:e])
    assert not flat[:b].any() and not flat[e:].any()
    assert not c[:b].any() and not c[e:].any() and not er[:b].any() and not er[e:].any()
    assert st["samples"] == int(c.sum())


def test_errors_and_fresh_state(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    good = [c.to_c() for c in fan(sc, 2)]
    adaptive_fields = {f for f, _ in _abi.rt_adaptive_params._fields_}

    def status(cams=good, n_views=None, view_base=0, w=W, h=H, null=(), null_cameras=False, **kw):
        arr = (_abi.rt_camera * max(len(cams), 1))(*cams)
        v = _abi.rt_views(len(cams) if n_views is None else n_views, view_base, None if null_cameras else arr)
        p = _abi.rt_render_params(w, h, 16, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
        a = _abi.rt_adaptive_params(4, 4, 0.05, 1e-3)
        for k, x in kw.items():
            setattr(a if k in adaptive_fields else p, k, x)
        args = {"p": C.byref(p), "v": C.byref(v), "a": C.byref(a)}
        for k in null:
            args[k] = None
        return L.rt_gpu_render_views_adaptive(rt._h, args["p"], args["v"], args["a"])

    assert status() == 0
    for k in ("p", "v", "a"):
        assert status(null=(k,)) == bad, k
    assert L.rt_gpu_render_views_adaptive(None, None, None, None) == bad
    assert status(n_views=0) == bad
    assert status(null_cameras=True) == bad
    for field, k in (("position", 0), ("right", 2), ("up", 1), ("forward", 2), ("fov_x", None)):
        for x in (float("nan"), float("inf")):
            c = _abi.rt_camera()
            C.memmove(C.byref(c), C.byref(good[0]), C.sizeof(c))
            if k is None:
                c.fov_x = x
            else:
                getattr(c, field)[k] = x
            assert status(cams=[good[1], c]) == bad, (field, x)
    top = (1 << 32) // (W * H)  # the 32-bit key: (view_base + n_views) * W * H <= 2^32
    assert status(view_base=top - 2) == 0
    assert status(view_base=top - 1) == bad and status(view_base=0xFFFFFFFF) == bad
    assert status(w=32768, h=32768) == bad  # 2 x 2^30 stacked pixels > 2^31 - 1 (the key bound holds)
    assert status(w=0) == bad
    for kw in ({"mode": _abi.RT_MODE_PRIMARY_IDS}, {"samples": 1}, {"sample_begin": 2}, {"sample_end": 8},
               {"flags": _abi.RT_FLAG_ACCUMULATE}, {"min_samples": 1}, {"step_samples": 0}, {"abs_floor": 0.0},
               {"abs_floor": -1.0}, {"rel_error": -1.0}, {"rel_error": float("nan")},
               {"pixel_begin": 10, "pixel_end": 5}, {"pixel_end": 2 * W * H + 1},
               {"max_paths_in_flight": 1024}):  # 2 x 96 x 64 pixels do not fit one batch of 1024 paths
        assert status(**kw) == bad, kw
    assert status(pixel_begin=W * H - 5, pixel_end=W * H + 5) == 0
    # the sums have per-pixel counts: accumulating onto them is refused
    assert status() == 0
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render(W, H, 8, seed=2, sample_begin=4, sample_end=8, accumulate=True)
    assert status() == 0
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_views(fan(sc, 2), W, H, 8, seed=2, sample_begin=4, sample_end=8, accumulate=True)
    # render_views without the flag is the render of a fresh handle, and leaves nothing adaptive
    assert status() == 0
    rt.render_views(fan(sc, 2), W, H, 6, seed=21)
    after, _ = rt.readback()
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
        rt.readback_adaptive()
    with gpu.RtGpu(1, 0) as fresh:
        fresh.upload_scene(sc)
        fresh.render_views(fan(sc, 2), W, H, 6, seed=21)
        assert np.array_equal(after, fresh.readback()[0])


def test_text_scene_is_refused(rt):
    from rt_b200 import textscene as T

    rt.upload_text_scene(T.load_npz(os.path.join(GOLDEN, "text", "scene-000.npz")))
    cam = rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_views_adaptive([cam], 16, 16, 8, 4, 4, 0.05)


def test_converged_after_round_zero_launches_at_most_two_rounds(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    rt.render_views_adaptive(cams, W, H, 4, 4, 4, 0.0, seed=1)
    one = rt.stats()["kernel_launches"]
    rt.render_views_adaptive(cams, W, H, 64, 4, 4, 1e9, seed=1)
    st = rt.stats()
    counts, _ = rt.readback_adaptive()
    print(f"launches: one round {one}, converged after round 0: {st['kernel_launches']}")
    assert np.all(counts == 4) and st["samples"] == 3 * W * H * 4
    assert one < st["kernel_launches"] <= 2 * one


def _n_dev():
    try:
        return gpu.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_dev() < 2, reason="needs >= 2 GPUs")
def test_two_devices_equal_one_device(golden_scene):
    sc = golden_scene("small_lights")
    cams = fan(sc, 3)
    out = []
    for n_gpus in (1, 2):
        with gpu.RtGpu(n_gpus, 0) as g:
            g.upload_scene(sc)
            g.render_views_adaptive(cams, W, H, 24, 4, 4, 0.05, seed=5)
            img, st = g.readback()
            counts, err = g.readback_adaptive()
            out.append((img, counts, err, st["samples"]))
    (a, ca, ea, sa), (b, cb, eb, sb) = out
    assert np.array_equal(a, b) and np.array_equal(ca, cb) and np.array_equal(ea, eb) and sa == sb
