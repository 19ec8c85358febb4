"""Multi-view rendering (rt_gpu_render_views) on the GPU.  V views of W x H are one stacked image of W x (V * H) pixels
and pixel p of view v is keyed (view_base + v) * W * H + p, so a one-view call with the scene's camera is rt_gpu_render
and view v of a call is a one-view call with view_base = v: the tests check both bit for bit, the per-view cameras
against the oracle, the stacked outputs, every error status, two devices and the CLI switch."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from conftest import GOLDEN
from views_scene import with_three_cameras, yawed

import rt_b200
from rt_b200 import _abi, gpu, host

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


def with_camera(scene, cam):
    """A shallow copy of `scene` whose own camera is `cam`"""
    s = copy.copy(scene)
    s.camera_position, s.camera_right, s.camera_up, s.camera_forward, s.fov_x = cam.position, cam.right, cam.up, cam.forward, cam.fov_x
    return s


@pytest.mark.parametrize("name", ["tiny", "small_lights", "tiny_env", "texmaps"])
def test_one_view_of_the_scene_camera_is_render(name, rt, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    rt.upload_scene(sc)
    rt.render(w, h, 8, seed=31)
    ref, st = rt.readback()
    ref8 = rt.readback_rgb8()
    ref_ids = rt.primary_ids(w, h)
    rt.render_views([sc.camera()], w, h, 8, seed=31)
    img, st_v = rt.readback()
    assert img.shape == (1, h, w, 3) and np.array_equal(img[0], ref)
    assert np.array_equal(rt.readback_rgb8()[0], ref8)
    assert st_v["samples"] == st["samples"] and st_v["kernel_launches"] == st["kernel_launches"]
    ids = rt.primary_ids(w, h, cameras=[sc.camera()])
    assert ids.shape == (1, h, w) and np.array_equal(ids[0], ref_ids)


def test_views_equal_one_view_calls(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 5)
    spp, seed = 8, 3
    for paths, exact in ((0, True), (4096, False)):  # 4096: pixel chunks of 4096 x 1 sample vs one-view batches
        rt.render_views(cams, W, H, spp, seed=seed, max_paths_in_flight=paths)
        many, st = rt.readback()
        assert many.shape == (5, H, W, 3) and st["samples"] == 5 * W * H * spp
        for v, cam in enumerate(cams):
            rt.render_views([cam], W, H, spp, seed=seed, view_base=v, max_paths_in_flight=paths)
            one = rt.readback()[0][0]
            if exact:
                assert np.array_equal(many[v], one), v
            else:
                assert np.allclose(many[v], one, rtol=2e-6, atol=1e-7), v
        if exact:
            ids = rt.primary_ids(W, H, cameras=cams)
            for v, cam in enumerate(cams):
                assert np.array_equal(ids[v], rt.primary_ids(W, H, cameras=[cam], view_base=v)[0]), v


@pytest.mark.parametrize("name", ["tiny", "small_lights"])
def test_view_ids_follow_the_oracle(name, rt, manifest, golden_scene):
    """Ids of every view against the oracle's ids of the scene with that camera (test_primary_ids_vs_reference's bound)."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    rt.upload_scene(sc)
    cams = fan(sc, 3, spread=12.0)
    ids = rt.primary_ids(w, h, cameras=cams)
    for v, cam in enumerate(cams):
        ref = O.primary_ids(with_camera(sc, cam), w, h)
        assert (ids[v] == ref).mean() >= 0.999, v
    assert not np.array_equal(ids[0], ids[2])


@pytest.mark.parametrize("name,tol_frac", [("tiny", 0.02), ("small_lights", 0.08)])
def test_other_camera_paths_follow_the_oracle(name, tol_frac, rt, manifest, golden_scene):
    """A one-view render (view_base = 0) of a camera that is not the scene's: path by path against the oracle's Philox
    mode on the scene with that camera, at test_paths_follow_oracle's bounds."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    cam = yawed(sc.camera(), 9.0)
    rt.upload_scene(sc)
    spp, seed = 32, 2024
    rt.render_views([cam], w, h, spp, seed=seed)
    img, st = rt.readback()
    img = img[0]
    ref, ost = O.render(with_camera(sc, cam), w, h, spp, rng_mode=O.RNG_PHILOX, seed=seed)
    rel = (np.abs(img - ref) / (np.abs(ref) + 1e-3)).max(axis=2)
    assert (rel > 1e-3).mean() <= tol_frac
    assert np.median(rel) < 2e-5
    assert abs(img.mean() - ref.mean()) < 5e-3 * ref.mean()
    assert abs(st["extension_rays"] - ost["extension_rays"]) <= 0.02 * ost["extension_rays"]


def test_views_are_independent(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    rt.render_views(cams, W, H, 6, seed=8)
    a, _ = rt.readback()
    cams[1] = yawed(sc.camera(), 33.0)
    rt.render_views(cams, W, H, 6, seed=8)
    b, _ = rt.readback()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])
    assert not np.array_equal(a[1], b[1])


def test_stacked_outputs_agree(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, 4)
    spp = 8
    rt.render_views(cams, W, H, spp, seed=12)
    full, st = rt.readback()
    rgb8 = rt.readback_rgb8()
    assert rgb8.shape == (4, H, W, 3)
    for v in range(4):
        assert np.abs(rgb8[v].astype(int) - host.tonemap_rgb8(full[v]).astype(int)).max() <= 1, v
    ptr, n = rt.accum_device_ptr()
    assert ptr and n == 4 * W * H * 4
    assert st["samples"] == 4 * W * H * spp
    # sample ranges accumulated into the same stacked sums
    rt.render_views(cams, W, H, spp, seed=12, sample_begin=0, sample_end=3)
    rt.render_views(cams, W, H, spp, seed=12, sample_begin=3, sample_end=spp, accumulate=True)
    parts, _ = rt.readback()
    assert np.allclose(parts, full, rtol=2e-6, atol=1e-7)
    # a pixel range that crosses from view 0 through view 1 into view 2
    b, e = W * H - 100, 2 * W * H + 37
    rt.render_views(cams, W, H, spp, seed=12, pixel_begin=b, pixel_end=e)
    part, st_p = rt.readback()
    flat, flat_full = part.reshape(-1, 3), full.reshape(-1, 3)
    assert np.array_equal(flat[b:e], flat_full[b:e])
    assert not flat[:b].any() and not flat[e:].any()
    assert st_p["samples"] == (e - b) * spp


def test_errors_and_fresh_state(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    good = [c.to_c() for c in fan(sc, 2)]

    def status(cams=good, n_views=None, view_base=0, w=W, h=H, flags=0, null_cameras=False):
        arr = (_abi.rt_camera * max(len(cams), 1))(*cams)
        v = _abi.rt_views(len(cams) if n_views is None else n_views, view_base, None if null_cameras else arr)
        p = _abi.rt_render_params(w, h, 4, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, flags, 0, 0)
        return L.rt_gpu_render_views(rt._h, C.byref(p), C.byref(v))

    assert status() == 0
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
    # the 32-bit key: (view_base + n_views) * W * H <= 2^32
    top = (1 << 32) // (W * H)  # 699050 views of 96 x 64 fit the key range
    assert status(view_base=top - 2) == 0
    assert status(view_base=top - 1) == bad
    assert status(view_base=0xFFFFFFFF) == bad
    # RT_FLAG_ACCUMULATE only onto the sums of the same width, height and n_views, in both directions
    acc = _abi.RT_FLAG_ACCUMULATE
    assert status() == 0 and status(flags=acc) == 0
    assert status(cams=good + good[:1], flags=acc) == bad
    assert status(w=W + 8, flags=acc) == bad
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render(W, H, 4, accumulate=True)  # after two views
    rt.render(W, H, 4)
    assert status(flags=acc) == bad  # two views onto one image
    assert status(cams=good[:1], flags=acc) == 0  # rt_gpu_render counts as one view of the same size
    rt.render(W, H, 4, accumulate=True)
    # nothing adaptive after views; rt_gpu_render after views is the render of a fresh handle
    assert status() == 0
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
        rt.readback_adaptive()
    rt.render(W, H, 6, seed=21)
    after, _ = rt.readback()
    assert after.shape == (H, W, 3)
    with gpu.RtGpu(1, 0) as fresh:
        fresh.upload_scene(sc)
        fresh.render(W, H, 6, seed=21)
        assert np.array_equal(after, fresh.readback()[0])


def test_text_scene_is_refused(rt):
    from rt_b200 import textscene as T

    ts = T.load_npz(os.path.join(GOLDEN, "text", "scene-000.npz"))
    rt.upload_text_scene(ts)
    cam = rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_views([cam], 16, 16, 4)


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
            g.render_views(cams, W, H, 8, seed=5)
            img, st = g.readback()
            g.render_views(cams, W, H, 1, seed=5)  # fewer samples than devices: the stacked image is split
            img1, _ = g.readback()
            out.append((img, img1, st["samples"]))
    (a, a1, sa), (b, b1, sb) = out
    assert np.allclose(a, b, rtol=2e-6, atol=1e-7) and sa == sb
    assert np.allclose(a1, b1, rtol=2e-6, atol=1e-7)


def _read_ppm(path):
    data = open(path, "rb").read()
    head, body = data.split(b"\n255\n", 1)
    w, h = map(int, head.split()[1:3])
    return np.frombuffer(body, np.uint8).reshape(h, w, 3)


def test_cli_renders_every_camera(scene_dir, tmp_path, monkeypatch):
    from rt_b200 import cli, gltf

    w, h, spp = 64, 48, 16
    path = with_three_cameras(scene_dir("tiny"), "tiny_three_cameras.gltf")
    monkeypatch.setenv("RT_CAMERAS", "all")
    assert cli.main(["prog", path, str(w), str(h), str(spp), str(tmp_path / "out.ppm")]) == 0
    outs = sorted(p.name for p in tmp_path.iterdir())
    assert outs == ["out_0.ppm", "out_1.ppm", "out_2.ppm"]
    sc = gltf.load_gltf(path, w / h)
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_views(sc.cameras, w, h, spp)
        means, _ = g.readback()
        for i in range(3):
            assert np.array_equal(_read_ppm(tmp_path / f"out_{i}.ppm"), host.tonemap_rgb8(means[i])), i
        g.render_views([sc.cameras[-1]], w, h, spp)  # the scene's own camera alone
        own, _ = g.readback()
    monkeypatch.delenv("RT_CAMERAS")
    assert cli.main(["prog", path, str(w), str(h), str(spp), str(tmp_path / "single.ppm")]) == 0
    assert np.array_equal(_read_ppm(tmp_path / "single.ppm"), host.tonemap_rgb8(own[0]))
    # RT_ADAPTIVE with RT_CAMERAS=all is refused
    monkeypatch.setenv("RT_CAMERAS", "all")
    monkeypatch.setenv("RT_ADAPTIVE", "0.05")
    assert cli.main(["prog", path, str(w), str(h), str(spp), str(tmp_path / "x.ppm")]) == 1
    assert not (tmp_path / "x_0.ppm").exists()
