"""Camera projections (rt_gpu_render_projected) on the GPU.  All-pinhole projections are rt_gpu_render_views /
rt_gpu_render_views_adaptive bit for bit and view v is a one-view call with view_base = v; the primary hits of the
other projections are those of the host's projected_ray traced on the host and by the float64 brute force; depth of
field, the equirectangular round trip through the environment map, every error status, two devices and the CLI."""
import ctypes as C

import numpy as np
import pytest

import hit_scenarios as hs
from projection_util import HostProjection, pixel_centre_rays, unit, with_camera_nodes
from views_scene import yawed

import rt_b200
from rt_b200 import _abi, gltf, gpu, host
from rt_b200._abi import Projection

pytestmark = pytest.mark.gpu

W, H = 96, 64  # whole 8 x 4 tiles: one tile never crosses a view


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hp():
    return HostProjection()


def fan(scene, n, spread=20.0):
    own = scene.camera()
    return [yawed(own, a) for a in np.linspace(-spread, spread, n)]


MIXED = [Projection.thin_lens(0.08, 3.0), Projection.orthographic(1.5, 1.0), Projection.equirect(), Projection.pinhole()]


@pytest.mark.parametrize("name", ["tiny", "small_lights", "tiny_env", "texmaps"])
def test_all_pinhole_is_render_views(name, rt, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    rt.upload_scene(sc)
    cams = fan(sc, 3)
    rt.render_views(cams, w, h, 8, seed=31)
    ref, st = rt.readback()
    ref8 = rt.readback_rgb8()
    ref_ids = rt.primary_ids(w, h, cameras=cams)
    for pin in (Projection.pinhole(), Projection.thin_lens(0.0, 2.0)):
        rt.render_projected(cams, [pin] * 3, w, h, 8, seed=31)
        img, st_p = rt.readback()
        assert img.shape == (3, h, w, 3) and np.array_equal(img, ref), pin
        assert np.array_equal(rt.readback_rgb8(), ref8)
        assert st_p["samples"] == st["samples"] and st_p["kernel_launches"] == st["kernel_launches"]
        assert np.array_equal(rt.primary_ids(w, h, cameras=cams, projections=[pin] * 3), ref_ids)
    # adaptive: rt_gpu_render_views_adaptive, counts and errors included
    rt.render_views_adaptive(cams, w, h, 24, 4, 4, 0.05, seed=7)
    ref, st = rt.readback()
    ref_c, ref_e = rt.readback_adaptive()
    rt.render_projected(cams, [Projection.pinhole()] * 3, w, h, 24, seed=7, adaptive=(4, 4, 0.05))
    img, st_p = rt.readback()
    c, e = rt.readback_adaptive()
    assert np.array_equal(img, ref) and np.array_equal(c, ref_c) and np.array_equal(e, ref_e)
    assert st_p["samples"] == st["samples"] and st_p["kernel_launches"] == st["kernel_launches"]


@pytest.mark.parametrize("adaptive", [None, (4, 4, 0.05)])
def test_view_v_is_a_one_view_call(adaptive, rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, len(MIXED))
    rt.render_projected(cams, MIXED, W, H, 16, seed=3, adaptive=adaptive)
    many, st = rt.readback()
    counts = rt.readback_adaptive()[0] if adaptive else None
    assert many.shape == (len(MIXED), H, W, 3) and np.isfinite(many).all()
    for v, (cam, pj) in enumerate(zip(cams, MIXED)):
        rt.render_projected([cam], [pj], W, H, 16, seed=3, view_base=v, adaptive=adaptive)
        assert np.array_equal(many[v], rt.readback()[0][0]), v
        if adaptive:
            assert np.array_equal(counts[v], rt.readback_adaptive()[0][0]), v
    # the projections change the image: no two views equal
    for a in range(len(MIXED)):
        for b in range(a + 1, len(MIXED)):
            assert not np.array_equal(many[a], many[b])


def test_accumulate_splits_the_sample_range(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    cams = fan(sc, len(MIXED))
    rt.render_projected(cams, MIXED, W, H, 8, seed=9)
    whole, _ = rt.readback()
    rt.render_projected(cams, MIXED, W, H, 8, seed=9, sample_begin=0, sample_end=3)
    rt.render_projected(cams, MIXED, W, H, 8, seed=9, sample_begin=3, sample_end=8, accumulate=True)
    split, st = rt.readback()
    assert st["samples"] == len(MIXED) * W * H * 5
    assert np.allclose(split, whole, rtol=1e-5, atol=1e-6)


def _aimed(tri):
    """A camera 1.5 box extents in front of the geometry, looking at its centre (as test_gpu_hits' views)."""
    lo, hi = tri.reshape(-1, 3).min(0).astype(np.float64), tri.reshape(-1, 3).max(0).astype(np.float64)
    c, ext = (lo + hi) / 2, max(float((hi - lo).max()), 1e-3)
    pos = (c + ext * np.array([0.3, 0.2, 1.5])).astype(np.float32)
    fwd = unit(c - pos.astype(np.float64))
    right = unit(np.cross(fwd, [0.0, 1.0, 0.0]))
    return rt_b200.Camera(pos, right, np.cross(right, fwd), fwd, 1.0), ext


@pytest.mark.parametrize("name", ["soup", "grid", "clusters", "far_3e3"])
def test_primary_hits_match_the_host_rays(name, rt, hp):
    """RT_MODE_PRIMARY_IDS of orthographic, equirectangular and thin-lens views against the same pixel-centre rays from
    the host's projected_ray, traced by hc_trace_rays and by the float64 brute force hc_brute_hits."""
    hc = hs.hostcheck()
    tri, _ = hs.make(name, 16)
    sc = hs.triangles_scene(tri)
    rt.upload_scene(sc)
    cam, ext = _aimed(tri)
    w, h = 64, 48
    # view 3: an orthographic view down -z from an axis-aligned camera, whose rays all have two zero components
    lo, hi = tri.reshape(-1, 3).min(0), tri.reshape(-1, 3).max(0)
    axis = rt_b200.Camera((lo + hi) / 2 + np.float32([0, 0, 1.5 * ext]), (1, 0, 0), (0, 1, 0), (0, 0, -1), 1.0)
    projs = [Projection.orthographic(0.6 * ext, 0.45 * ext), Projection.equirect(), Projection.thin_lens(0.05 * ext, 1.2 * ext),
             Projection.orthographic(0.6 * ext, 0.45 * ext)]
    cams = [cam, cam, cam, axis]
    ids = rt.primary_ids(w, h, cameras=cams, projections=projs)
    pin = rt.primary_ids(w, h, cameras=[cam], projections=[Projection.pinhole()])[0]
    assert np.array_equal(ids[2], pin), "pixel-centre rays pass through the lens centre: the pinhole's hits"
    for v in (0, 1, 3):
        pj = projs[v]
        rays = np.ascontiguousarray(pixel_centre_rays(hp, cams[v], pj, w, h))
        n = len(rays)
        ie, iq = np.zeros(n, np.int32), np.zeros(n, np.int32)
        te, tq = np.zeros(n, np.float32), np.zeros(n, np.float32)
        d = sc.desc()
        hc.hc_set_rebuild(1)  # the scene has no host tree: pack with the library's builder
        try:
            assert hc.hc_trace_rays(C.byref(d), C.c_uint64(n), hs._ptr(rays), hs._ptr(ie), hs._ptr(te), hs._ptr(iq), hs._ptr(tq)) == 0
        finally:
            hc.hc_set_rebuild(0)
        got = ids[v].reshape(-1)
        exp = hs.Expected(hc, tri, rays, sc.eps)
        wrong = exp.wrong(got)
        differ = got != ie
        print(f"{name} {Projection.NAMES[pj.kind]}: {(got >= 0).mean():.3f} of the pixels hit, {int(differ.sum())} differ from "
              f"hc_trace_rays, decidable {exp.dec.mean():.3f}, wrong {int(wrong.sum())}")
        assert (got >= 0).mean() > 0.005
        assert not wrong.any(), f"{int(wrong.sum())} decidable rays miss their nearest hit"
        # host and device evaluate projected_ray in the same float32 operations; a contracted multiply-add on the device
        # can move a ray by an ulp, which only matters for rays that graze an edge (not decidable)
        assert not (differ & exp.dec & (exp.ties <= 1)).any()


def _checker_scene(depth, n=16, half=2.5):
    """Quads of a checkerboard (every other square present) in the plane z = -depth, facing +z, in front of the
    constant white sky; camera at the origin looking down -z."""
    quads = []
    s = 2 * half / n
    for i in range(n):
        for j in range(n):
            if (i + j) % 2 == 0:
                x0, y0 = -half + i * s, -half + j * s
                a, b, c, d = [x0, y0, -depth], [x0 + s, y0, -depth], [x0 + s, y0 + s, -depth], [x0, y0 + s, -depth]
                quads += [[a, b, c], [a, c, d]]
    sc = hs.triangles_scene(np.array(quads, np.float32))
    sc.camera_position = np.zeros(3, np.float32)
    return sc


def _gradient(img):
    y = img.mean(-1)
    return float(np.abs(np.diff(y, axis=0)).mean() + np.abs(np.diff(y, axis=1)).mean())


def test_depth_of_field(rt):
    """Focused on the plane, a thin lens renders what the pinhole renders, within 1.5 x the seed-to-seed noise of the
    pinhole; focused elsewhere it blurs the checker edges (lower mean gradient); over many spp its mean image does not
    depend on the lens samples' seed beyond the noise."""
    depth, w, h, spp = 4.0, 64, 64, 256
    sc = _checker_scene(depth)
    rt.upload_scene(sc)
    cam = sc.camera()

    def render(pj, seed):
        rt.render_projected([cam], [pj], w, h, spp, seed=seed)
        return rt.readback()[0][0].astype(np.float64)

    pin_a, pin_b = render(Projection.pinhole(), 1), render(Projection.pinhole(), 2)
    noise = np.abs(pin_a - pin_b).mean()
    focused = render(Projection.thin_lens(0.15, depth), 1)
    off = render(Projection.thin_lens(0.15, depth / 3), 1)
    off_b = render(Projection.thin_lens(0.15, depth / 3), 2)
    print(f"noise {noise:.4f}, focused - pinhole {np.abs(focused - pin_a).mean():.4f}; gradients: pinhole {_gradient(pin_a):.4f}, "
          f"focused {_gradient(focused):.4f}, off focus {_gradient(off):.4f}")
    assert np.abs(focused - pin_a).mean() <= 1.5 * noise
    assert _gradient(off) < 0.6 * _gradient(pin_a)
    assert abs(_gradient(focused) - _gradient(pin_a)) < 0.15 * _gradient(pin_a)
    diff = off - off_b
    assert abs(diff.mean()) <= 4 * diff.std() / np.sqrt(diff.size)
    assert np.abs(diff).mean() <= 1.5 * noise


def test_equirect_round_trip_through_the_environment_map(rt, golden_scene):
    """An empty world (one invisible far triangle) with tiny_env's 64 x 32 map: a 64 x 32 equirectangular view with
    forward = +x, right = +z, up = +y reproduces the map.  The pixel jitter averages the bilinear lookup over +-0.5 texel,
    i.e. the map filtered with [1/8, 3/4, 1/8] along x and y; the rows at the poles are left out."""
    env = golden_scene("tiny_env")
    sc = hs.triangles_scene(np.array([[[1e4, 0, 0], [1e4, 1e-3, 0], [1e4, 0, 1e-3]]], np.float32) * -1)
    sc.materials, sc.textures, sc.texels, sc.env_texture = env.materials, env.textures, env.texels, env.env_texture
    sc.bg_color = env.bg_color
    rt.upload_scene(sc)
    tw, th = (int(x) for x in env.textures[env.env_texture - 1][["width", "height"]])
    cam = rt_b200.Camera([0, 0, 0], [0, 0, 1], [0, 1, 0], [1, 0, 0], 1.0)
    rt.render_projected([cam], [Projection.equirect()], tw, th, 1024, seed=4)
    img = rt.readback()[0][0].astype(np.float64)
    tex = env.texels[:tw * th * 4].reshape(th, tw, 4)[..., :3].astype(np.float64)
    lin = (tex / 255.0) ** 2.2 * env.bg_color.astype(np.float64)
    k = (0.125, 0.75, 0.125)
    fx = k[0] * np.roll(lin, 1, 1) + k[1] * lin + k[2] * np.roll(lin, -1, 1)
    expect = k[0] * np.roll(fx, 1, 0) + k[1] * fx + k[2] * np.roll(fx, -1, 0)
    inner = slice(1, th - 1)
    err = np.abs(img[inner] - expect[inner])
    print(f"equirect round trip: mean |err| {err.mean():.5f}, max {err.max():.5f}, mean value {expect[inner].mean():.4f}")
    assert err.mean() <= 0.02 * expect[inner].mean() + 1e-3
    assert np.quantile(err, 0.99) <= 0.1 * expect[inner].max() + 1e-3
    # the unfiltered map is further away than the filtered one: the lookup is centred on texel (i, j), not shifted
    assert err.mean() < np.abs(img[inner] - np.roll(expect, 1, 1)[inner]).mean()


def test_errors_and_state(rt, golden_scene):
    sc = golden_scene("small_lights")
    rt.upload_scene(sc)
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    cams = [c.to_c() for c in fan(sc, 2)]

    def status(projs, adaptive=None, null=(), **kw):
        arr = (_abi.rt_camera * 2)(*cams)
        pa = (_abi.rt_projection * 2)(*[p if isinstance(p, _abi.rt_projection) else p.to_c() for p in projs])
        v = _abi.rt_views(2, 0, arr)
        p = _abi.rt_render_params(W, H, 16, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
        for k, x in kw.items():
            setattr(p, k, x)
        a = None if adaptive is None else C.byref(_abi.rt_adaptive_params(*adaptive))
        args = {"p": C.byref(p), "v": C.byref(v), "j": pa}
        for k in null:
            args[k] = None
        return L.rt_gpu_render_projected(rt._h, args["p"], args["v"], args["j"], a)

    good = [Projection.thin_lens(0.1, 3.0), Projection.orthographic(1.0, 0.5)]
    rt.render_projected(fan(sc, 2), good, W, H, 6, seed=21)
    before, _ = rt.readback()
    inf, nan = float("inf"), float("nan")
    refused = [_abi.rt_projection(4, 0, 0, 0, 0), _abi.rt_projection(0xFFFFFFFF, 0, 0, 0, 0),
               _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, -0.1, 3, 0, 0), _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, 0.1, 0, 0, 0),
               _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, 0.1, -2, 0, 0), _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, nan, 3, 0, 0),
               _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, 0.1, inf, 0, 0), _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, inf, 3, 0, 0),
               _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, 0, 0, 0, 1), _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, 0, 0, 1, -1),
               _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, 0, 0, nan, 1), _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, 0, 0, 1, inf)]
    for r in refused:
        for adaptive in (None, (4, 4, 0.05, 1e-3)):
            assert status([good[0], r], adaptive) == bad, (r.kind, r.aperture_radius, r.focus_distance, r.half_width, r.half_height)
            assert "rt_gpu_render_projected" in L.rt_gpu_last_error().decode()
    # a refused call leaves the last render readable and unchanged
    assert np.array_equal(rt.readback()[0], before)
    # fields a kind does not use are ignored, even when non-finite; a zero aperture needs no focus distance
    ignored = [_abi.rt_projection(_abi.RT_PROJ_PINHOLE, nan, -1, inf, -1), _abi.rt_projection(_abi.RT_PROJ_EQUIRECT, -1, nan, 0, 0),
               _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, 0, 0, nan, -1), _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, -1, nan, 1, 1)]
    for r in ignored:
        assert status([good[0], r]) == 0, r.kind
    # the refusals of the view calls
    for k in ("p", "v", "j"):
        assert status(good, null=(k,)) == bad, k
    assert L.rt_gpu_render_projected(None, None, None, None, None) == bad
    for kw in ({"width": 0}, {"samples": 0}, {"sample_begin": 9, "sample_end": 4}, {"pixel_begin": 10, "pixel_end": 5},
               {"pixel_end": 2 * W * H + 1}):
        assert status(good, **kw) == bad, kw
    for kw in ({"mode": _abi.RT_MODE_PRIMARY_IDS}, {"samples": 1}, {"sample_end": 8}, {"flags": _abi.RT_FLAG_ACCUMULATE}):
        assert status(good, (4, 4, 0.05, 1e-3), **kw) == bad, kw
    assert status(good, (1, 4, 0.05, 1e-3)) == bad and status(good, (4, 4, 0.05, 0.0)) == bad
    # after an adaptive projected render the sums have counts: accumulating onto them is refused
    assert status(good, (4, 4, 0.05, 1e-3)) == 0
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_projected(fan(sc, 2), good, W, H, 8, seed=2, sample_begin=4, sample_end=8, accumulate=True)
    # without the flag a render is the render of a fresh handle
    rt.render_projected(fan(sc, 2), good, W, H, 6, seed=21)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
        rt.readback_adaptive()
    assert np.array_equal(rt.readback()[0], before)


def _n_dev():
    try:
        return gpu.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_dev() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("adaptive", [None, (4, 4, 0.05)])
def test_two_devices_equal_one_device(adaptive, golden_scene):
    sc = golden_scene("small_lights")
    cams = fan(sc, len(MIXED))
    out = []
    for n_gpus in (1, 2):
        with gpu.RtGpu(n_gpus, 0) as g:
            g.upload_scene(sc)
            g.render_projected(cams, MIXED, W, H, 24, seed=5, adaptive=adaptive)
            img, st = g.readback()
            out.append((img, g.readback_adaptive()[0] if adaptive else None, st["samples"]))
    (a, ca, sa), (b, cb, sb) = out
    assert sa == sb and np.array_equal(ca, cb)
    if adaptive:
        assert np.array_equal(a, b)
    else:  # the sample split sums in another order
        assert np.allclose(a, b, rtol=1e-5, atol=1e-6)


def _read_ppm(path):
    data = open(path, "rb").read()
    w, h = (int(x) for x in data.split(b"\n")[1].split())
    return np.frombuffer(data.split(b"\n255\n", 1)[1], np.uint8).reshape(h, w, 3)


def test_cli_projection(scene_dir, tmp_path, monkeypatch):
    from rt_b200 import cli

    w, h, spp = 64, 48, 16
    src = scene_dir("tiny")
    sc = gltf.load_gltf(src, w / h)
    ortho = Projection.orthographic(1.5, 1.125)
    monkeypatch.setenv("RT_PROJECTION", "ortho:1.5:1.125")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "o.ppm")]) == 0
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_projected([sc.camera()], [ortho], w, h, spp, max_paths_in_flight=128 << 20)
        mean, _ = g.readback()
    assert np.array_equal(_read_ppm(tmp_path / "o.ppm"), host.tonemap_rgb8(mean[0]))
    monkeypatch.setenv("RT_PROJECTION", "fisheye")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "x.ppm")]) == 1
    assert not (tmp_path / "x.ppm").exists()
    # RT_CAMERAS=all renders each camera node with its own projection
    monkeypatch.delenv("RT_PROJECTION")
    own = sc.cameras[-1]
    import json
    with open(src) as f:
        doc = json.load(f)
    persp = doc["cameras"][next(n for n in doc["nodes"] if "camera" in n)["camera"]]
    path = with_camera_nodes(src, "tiny_ortho_cli.gltf", [({"type": "orthographic", "orthographic": {"xmag": 1.5, "ymag": 1.125,
                                                            "znear": 0.01, "zfar": 100}}, own.position), (persp, own.position)])
    both = gltf.load_gltf(path, w / h)
    assert both.projections == [ortho, Projection.pinhole()]
    monkeypatch.setenv("RT_CAMERAS", "all")
    assert cli.main(["prog", path, str(w), str(h), str(spp), str(tmp_path / "v.ppm")]) == 0
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(both)
        g.render_projected(both.cameras, both.projections, w, h, spp, max_paths_in_flight=128 << 20)
        means, _ = g.readback()
    for i in range(2):
        assert np.array_equal(_read_ppm(tmp_path / f"v_{i}.ppm"), host.tonemap_rgb8(means[i])), i
