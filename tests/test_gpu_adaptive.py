"""Adaptive sampling (rt_gpu_render_adaptive) on the GPU.  Every pixel receives the sample prefix [0, n_p) and Philox
is keyed by (pixel, sample), so an adaptive image is, pixel by pixel, a fixed render truncated at that pixel's count:
the tests compare it bit for bit with fixed renders, check the stopping rule against its definition and the moments
against a host computation, and hold the result to the same statistical-parity bounds as the fixed render."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import golden_array, rel_mse

import rt_b200  # noqa: F401
from rt_b200 import _abi, gpu, host

pytestmark = pytest.mark.gpu

W, H = 96, 64  # whole 8 x 4 tiles: the first active list is in k_generate's tile order


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


def _median_target(rt, seed):
    """The stopping target taken from the data: the median err after one 4-sample round."""
    rt.render_adaptive(W, H, 4, 4, 4, 0.0, seed=seed)
    _, err = rt.readback_adaptive()
    return float(np.median(err))


def _fixed_in_steps(rt, n, seed, first=4, step=4):
    """samples [0, first), [first, first + step) ... [.., n) as accumulated fixed renders of an n-spp image"""
    rt.render(W, H, n, seed=seed, sample_begin=0, sample_end=min(first, n))
    s = first
    while s < n:
        rt.render(W, H, n, seed=seed, sample_begin=s, sample_end=min(s + step, n), accumulate=True)
        s += step
    return rt.readback()[0]


def test_adaptive_equals_truncated_fixed_renders(rt, golden_scene):
    rt.upload_scene(golden_scene("small_lights"))
    seed, lo, step, hi = 5, 4, 4, 24
    target = _median_target(rt, seed)
    rt.render_adaptive(W, H, hi, lo, step, target, seed=seed)
    img, st = rt.readback()
    counts, err = rt.readback_adaptive()
    values = sorted(set(counts.ravel().tolist()))
    print(f"target {target:.4f}: counts {values}, {counts.sum() / (W * H * hi):.3f} of the maximum traced")
    assert len(values) >= 3 and lo in values and hi in values
    # the stopping invariant
    assert all((v - lo) % step == 0 or v == hi for v in values) and min(values) >= lo and max(values) <= hi
    assert np.all(err[counts < hi] <= target)
    assert np.all(counts[err > target] == hi)
    assert st["samples"] == int(counts.sum())
    # bit identity: every pixel whose count is n equals the fixed render of n samples made of the same sample ranges
    for n in values:
        fixed = _fixed_in_steps(rt, n, seed)
        sel = counts == n
        assert np.array_equal(img[sel], fixed[sel]), n


def test_target_zero_in_one_round_is_the_fixed_render(rt, golden_scene):
    rt.upload_scene(golden_scene("small_lights"))
    rt.render(W, H, 6, seed=9)
    fixed, st = rt.readback()
    fixed8 = rt.readback_rgb8()
    rt.render_adaptive(W, H, 6, 6, 1, 0.0, seed=9)
    img, st2 = rt.readback()
    counts, _ = rt.readback_adaptive()
    assert np.array_equal(img, fixed) and np.all(counts == 6)
    assert np.array_equal(rt.readback_rgb8(), fixed8)
    assert st2["samples"] == st["samples"] == W * H * 6


def test_error_map_matches_host_moments(rt, golden_scene):
    """min 2, step 1, max 8 at target 0: every pixel runs to 8; its err against float64 moments of 8 one-sample
    fixed renders."""
    rt.upload_scene(golden_scene("small_lights"))
    seed, n, floor = 13, 8, 1e-3
    ys = []
    for s in range(n):
        rt.render(W, H, 1, seed=seed, sample_begin=s, sample_end=s + 1)
        ys.append(rt.readback()[0].astype(np.float64).sum(axis=2) / 3.0)
    y = np.stack(ys)
    S, Q = y.sum(axis=0), (y * y).sum(axis=0)
    m = S / n
    var = np.maximum(Q / n - m * m, 0.0) * n / (n - 1)
    want = np.sqrt(var / n) / (m + floor)
    rt.render_adaptive(W, H, n, 2, 1, 0.0, abs_floor=floor, seed=seed)
    counts, err = rt.readback_adaptive()
    assert np.all(counts == n)
    # Q is summed in float32 on the device: a variance at the rounding level of Q / n (e.g. the sky's) is noise
    atol = np.sqrt(16 * 2.0 ** -23 * (Q / n) / n) / (m + floor)
    ok = np.abs(err - want) <= 1e-4 * want + atol
    print(f"err: {ok.mean() * 100:.3f} % within tolerance, max |diff| {np.abs(err - want).max():.3g}")
    assert ok.all()


@pytest.mark.parametrize("name,target", [("tiny", 0.005), ("small_lights", 0.005), ("texmaps", 0.005), ("big_lights", 0.005)])
def test_statistical_parity_adaptive(name, target, rt, manifest, golden_scene, big_scene):
    """The north-star bounds of test_statistical_parity_small with max spp = 8 x hi_spp and a relative-error target of
    0.5 % (min = step = max / 16): relMSE < 1e-3 against the reference's hi-spp render, 8-bit MAE <= 1.  This also
    bounds the bias of stopping on a noise estimate."""
    m = manifest["scenes"][name]
    w, h, hi = m["width"], m["height"], m["hi_spp"]
    spp = 8 * hi
    rt.upload_scene(big_scene if name == "big_lights" else golden_scene(name))
    rt.render_adaptive(w, h, spp, spp // 16, spp // 16, target, seed=77)
    img, st = rt.readback()
    a = golden_array(f"{name}_refhi_a.f32", np.float32, (h, w, 3))
    err = rel_mse(img, a)
    mae = np.abs(host.tonemap_rgb8(img).astype(np.int32) - host.tonemap_rgb8(a).astype(np.int32)).mean()
    frac = st["samples"] / (w * h * spp)
    print(f"{name}: relMSE {err}, 8-bit MAE {mae:.3f}, {frac:.3f} of the maximum samples traced")
    assert np.all(err < 1e-3), err
    assert mae <= 1.0, mae
    assert st["samples"] < w * h * spp


def test_pixel_range_errors_and_fresh_state(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    b, e = 17 * W + 23, 41 * W + 5  # not on row boundaries
    rt.render(W, H, 8, seed=4, pixel_begin=b, pixel_end=e)
    fixed, _ = rt.readback()
    rt.render_adaptive(W, H, 8, 8, 1, 0.0, seed=4, pixel_begin=b, pixel_end=e)
    img, st = rt.readback()
    counts, err = rt.readback_adaptive()
    flat_c, flat_e = counts.ravel(), err.ravel()
    assert np.array_equal(img, fixed)
    assert not img.reshape(-1, 3)[:b].any() and not img.reshape(-1, 3)[e:].any()
    assert not flat_c[:b].any() and not flat_c[e:].any() and np.all(flat_c[b:e] == 8)
    assert not flat_e[:b].any() and not flat_e[e:].any()
    assert st["samples"] == (e - b) * 8

    L = gpu.lib()

    adaptive_fields = {f for f, _ in _abi.rt_adaptive_params._fields_}

    def status(**kw):  # rt_gpu_render_adaptive with one field of the parameters changed
        params = _abi.rt_render_params(W, H, 16, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
        adapt = _abi.rt_adaptive_params(4, 4, 0.05, 1e-3)
        for k, v in kw.items():
            setattr(adapt if k in adaptive_fields else params, k, v)
        return L.rt_gpu_render_adaptive(rt._h, C.byref(params), C.byref(adapt))

    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    assert status() == 0
    for kw in ({"sample_begin": 2}, {"sample_end": 8}, {"flags": _abi.RT_FLAG_ACCUMULATE}, {"mode": _abi.RT_MODE_PRIMARY_IDS},
               {"min_samples": 1}, {"step_samples": 0}, {"abs_floor": 0.0}, {"abs_floor": -1.0},
               {"max_paths_in_flight": 1024}):  # 96 x 64 pixels do not fit one batch of 1024 paths
        assert status(**kw) == bad, kw
    # accumulating onto adaptive sums is refused; readback_adaptive after a fixed render has nothing to return
    rt.render_adaptive(W, H, 8, 4, 4, 0.05, seed=2)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render(W, H, 8, seed=2, sample_begin=4, sample_end=8, accumulate=True)
    # a fixed render after an adaptive one is the render of a fresh handle
    rt.render(W, H, 6, seed=21)
    after, _ = rt.readback()
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
        rt.readback_adaptive()
    with gpu.RtGpu(1, 0) as fresh:
        fresh.upload_scene(sc)
        fresh.render(W, H, 6, seed=21)
        assert np.array_equal(after, fresh.readback()[0])


def test_text_scene_is_refused(rt):
    from rt_b200 import textscene as T
    from conftest import GOLDEN

    ts = T.load_npz(os.path.join(GOLDEN, "text", "scene-000.npz"))
    rt.upload_text_scene(ts)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_adaptive(16, 16, 8, 4, 4, 0.05)


def test_converged_after_round_zero_launches_at_most_two_rounds(rt, golden_scene):
    """Round r + 2 is enqueued only after round r's active count arrived: with every pixel done after round 0 the
    render launches round 1 (empty) and stops."""
    rt.upload_scene(golden_scene("small_lights"))
    rt.render_adaptive(W, H, 4, 4, 4, 0.0, seed=1)
    one = rt.stats()["kernel_launches"]
    rt.render_adaptive(W, H, 64, 4, 4, 1e9, seed=1)
    st = rt.stats()
    counts, _ = rt.readback_adaptive()
    print(f"launches: one round {one}, converged after round 0: {st['kernel_launches']}")
    assert np.all(counts == 4) and st["samples"] == W * H * 4
    assert one < st["kernel_launches"] <= 2 * one


def _n_dev():
    try:
        return gpu.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_dev() < 2, reason="needs >= 2 GPUs")
def test_two_devices_equal_one_device(golden_scene):
    sc = golden_scene("small_lights")
    out = []
    for n_gpus in (1, 2):
        with gpu.RtGpu(n_gpus, 0) as g:
            g.upload_scene(sc)
            g.render_adaptive(W, H, 24, 4, 4, 0.05, seed=5)
            img, st = g.readback()
            counts, err = g.readback_adaptive()
            out.append((img, counts, err, st["samples"]))
    (a, ca, ea, sa), (b, cb, eb, sb) = out
    assert np.array_equal(a, b) and np.array_equal(ca, cb) and np.array_equal(ea, eb) and sa == sb


def test_cli_adaptive_switch(scene_dir, tmp_path, manifest, capsys, monkeypatch):
    """RT_ADAPTIVE=<rel_error>: the 4th argument is the maximum spp; the PPM stays within the fixed CLI test's bound of
    the stored 16 384-spp reference render."""
    from rt_b200 import cli

    w, h, spp = 64, 48, 4096
    golden = host.tonemap_rgb8(golden_array("tiny_refhi_a.f32", np.float32, (h, w, 3)))
    monkeypatch.setenv("RT_ADAPTIVE", "0.005")
    assert cli.main(["prog", scene_dir("tiny"), str(w), str(h), str(spp), str(tmp_path / "o.ppm")]) == 0
    data = open(tmp_path / "o.ppm", "rb").read()
    img = np.frombuffer(data.split(b"\n255\n", 1)[1], np.uint8).reshape(h, w, 3)
    mae = np.abs(img.astype(int) - golden.astype(int)).mean()
    msg = capsys.readouterr().err
    print(msg, f"MAE {mae:.3f}")
    assert "samples traced" in msg
    assert mae < 1.0, mae
