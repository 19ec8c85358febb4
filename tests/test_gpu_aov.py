"""AOV render (rt_gpu_render_aov / rt_gpu_readback_aov) on the GPU: at ray depth 1 under a black sky the emission AOV is
the beauty render's mean bit for bit (scene camera, views, projections); pixel-centre AOVs against the reference's pinned
hit data; alpha walks at the scenes' own ray depth against the host statement hc_aov; the view / projection identities;
the beauty state left alone; every refusal; the 8-wide library; two devices; both CLIs."""
import copy
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, golden_array
from views_scene import yawed

from rt_b200 import _abi, gltf, gpu, host, pfm
from rt_b200._abi import Projection

pytestmark = pytest.mark.gpu

NAMES = ("albedo", "normal", "emission", "depth", "coverage")
LENSES = [Projection.thin_lens(0.08, 3.0), Projection.orthographic(1.5, 1.0), Projection.equirect()]
WHICH_LIB = os.path.basename(os.environ.get("RT_GPU_LIB", "librt_gpu.so"))


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hc():
    L = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libaovcheck.so"))  # libhostcheck.so + hc_aov
    L.hc_aov.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]
    return L


def fan(scene, n, spread=20.0):
    own = scene.camera()
    return [yawed(own, a) for a in np.linspace(-spread, spread, n)]


def black_sky_depth1(sc):
    s = copy.copy(sc)
    s.ray_depth = 1
    s.bg_color = np.zeros(3, np.float32)
    return s


def same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in NAMES)


@pytest.mark.parametrize("name", ["tiny", "small_lights", "texmaps", "texall"])
def test_emission_at_depth_one_is_the_beauty_mean(name, rt, manifest, golden_scene):
    """Identity 1: ray depth 1, black sky, the same params in one batch: emission == rgb_mean bit for bit, through
    rt_gpu_render, rt_gpu_render_views (3 views) and rt_gpu_render_projected (thin lens, orthographic, equirect)."""
    m = manifest["scenes"][name]
    w, h, spp = m["width"], m["height"], 8
    sc = black_sky_depth1(golden_scene(name))
    rt.upload_scene(sc)
    rt.render(w, h, spp, seed=17)
    ref, _ = rt.readback()
    rt.render_aov(w, h, spp, seed=17)
    a = rt.readback_aov()
    assert a["emission"].shape == (h, w, 3) and a["depth"].shape == (h, w)
    assert np.array_equal(a["emission"], ref)
    cams = fan(sc, 3)
    rt.render_views(cams, w, h, spp, seed=17)
    ref, _ = rt.readback()
    rt.render_aov(w, h, spp, seed=17, cameras=cams)
    assert np.array_equal(rt.readback_aov()["emission"], ref)
    rt.render_projected(cams, LENSES, w, h, spp, seed=17)
    ref, _ = rt.readback()
    rt.render_aov(w, h, spp, seed=17, cameras=cams, projections=LENSES)
    a = rt.readback_aov()
    assert a["emission"].shape == (3, h, w, 3) and np.array_equal(a["emission"], ref)


@pytest.mark.parametrize("name", ["tiny", "small_lights", "texmaps", "texall", "tiny_lt", "small_lights_lt"])
def test_pixel_centres_match_the_reference_hit_data(name, rt, manifest, golden_scene):
    """centre=True against the reference's pinned *_hitinfo.f32 on hit pixels whose first surface has alpha 1, with the
    tolerances of test_device_hit_data_matches_reference; coverage == (RT_MODE_PRIMARY_IDS ids >= 0) everywhere."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    rt.upload_scene(golden_scene(name))
    ids = rt.primary_ids(w, h)
    rt.render_aov(w, h, 1, centre=True)
    a = rt.readback_aov()
    ref = golden_array(f"{name}_hitinfo.f32", np.float32, (h, w, 18))
    ref_ids = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    ok = (ref_ids >= 0) & (ids >= 0) & (ref[..., 10] == 1.0)
    assert ok.sum() > 0.2 * w * h
    got = np.concatenate([a["depth"][..., None], a["normal"], a["albedo"], a["emission"]], axis=2)[ok]
    want = ref[ok][:, np.r_[0, 4:7, 7:10, 11:14]]
    diff = np.abs(got - want)
    diff[:, 0] /= np.maximum(want[:, 0], 1.0)  # t relative
    assert np.quantile(diff, 0.999) < 1e-4 and diff.max() < 5e-3
    # misses, and hits whose first surface has alpha 1: coverage is the id render's ids >= 0
    decided = (ids < 0) | ok
    assert np.array_equal(a["coverage"][decided] == 1.0, ids[decided] >= 0)
    assert np.all((a["coverage"] == 0) | (a["coverage"] == 1))


# the fractions of the path-by-path parity tests (test_gpu_parity.py); texall's 0.6 there comes from its near-mirrors'
# BRDF, which the walk does not evaluate
@pytest.mark.parametrize("name,tol_frac", [("tiny", 0.02), ("small_lights", 0.08), ("texmaps", 0.02), ("texall", 0.05)])
def test_alpha_walk_matches_the_host_statement(name, tol_frac, rt, hc, manifest, golden_scene):
    """The scenes' own ray depth, 1 spp: every channel agrees with hc_aov per pixel except on a small fraction (host and
    device trees can break ties differently, and a pass-through origin may differ in its last bit)."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    rt.upload_scene(sc)
    rt.render_aov(w, h, 1, seed=9)
    a = rt.readback_aov()
    d = sc.desc()
    out = np.zeros((h, w, 11), np.float32)
    assert hc.hc_aov(C.byref(d), w, h, 1, 9, 0, out.ctypes.data_as(C.c_void_p)) == 0
    dev = np.concatenate([a["albedo"], a["normal"], a["emission"], a["depth"][..., None], a["coverage"][..., None]], axis=2)
    close = np.isclose(dev, out, rtol=1e-4, atol=1e-5).all(axis=2)
    frac = 1.0 - close.mean()
    print(f"{name} [{WHICH_LIB}]: {frac:.4f} of pixels differ from hc_aov; coverage {a['coverage'].mean():.4f} "
          f"(host {out[..., 10].mean():.4f})")
    assert frac <= tol_frac
    assert abs(a["coverage"].mean() - out[..., 10].mean()) <= tol_frac


def test_view_and_projection_identities(rt, golden_scene):
    """Identity 2: view v of a V-view call == a one-view call with view_base = v; all-pinhole projections == none;
    views == NULL == one view of the scene camera; two renders of the same arguments are identical."""
    sc = golden_scene("small_lights")
    w, h, spp = 48, 32, 6
    rt.upload_scene(sc)
    cams = fan(sc, 4)
    rt.render_aov(w, h, spp, seed=3, cameras=cams, projections=LENSES + [Projection.pinhole()])
    multi = rt.readback_aov()
    for v in range(4):
        rt.render_aov(w, h, spp, seed=3, cameras=[cams[v]], projections=[(LENSES + [Projection.pinhole()])[v]], view_base=v)
        one = rt.readback_aov()
        assert all(np.array_equal(multi[k][v], one[k][0]) for k in NAMES), v
    rt.render_aov(w, h, spp, seed=3, cameras=cams)
    plain = rt.readback_aov()
    rt.render_aov(w, h, spp, seed=3, cameras=cams, projections=[Projection.pinhole()] * 4)
    assert same(plain, rt.readback_aov())
    rt.render_aov(w, h, spp, seed=3)
    own = rt.readback_aov()
    rt.render_aov(w, h, spp, seed=3, cameras=[sc.camera()])
    assert all(np.array_equal(own[k], v[0]) for k, v in rt.readback_aov().items())
    rt.render_aov(w, h, spp, seed=3)
    assert same(own, rt.readback_aov())
    # a pixel range: the rest reads 0, the range is the full render's
    rt.render_aov(w, h, spp, seed=3, pixel_begin=100, pixel_end=700)
    part = rt.readback_aov()
    for k in NAMES:
        flat, ref = part[k].reshape(w * h, -1), own[k].reshape(w * h, -1)
        assert np.array_equal(flat[100:700], ref[100:700]) and not flat[:100].any() and not flat[700:].any()
    st = rt.aov_stats()
    assert st["samples"] == 600 * spp and st["extension_rays"] >= st["samples"] and st["kernel_launches"] > 0 and st["render_ms"] > 0


def _ids(rt):
    w, h, _ = rt._last
    ids = np.empty(rt._shape(), np.int32)
    assert gpu.lib().rt_gpu_readback(rt._h, None, ids.ctypes.data_as(C.c_void_p), None) == 0
    return ids


def test_beauty_state_is_left_alone(rt, golden_scene):
    """Identity 3: beauty means, rgb8, stats, ids and adaptive counts / errors read the same before and after an AOV
    render; render_projected followed by render_aov gives the image and its matching buffers on one handle."""
    sc = golden_scene("texmaps")
    w, h = 40, 32
    rt.upload_scene(sc)
    cams = fan(sc, 2)
    rt.render_projected(cams, LENSES[:2], w, h, 8, seed=4)
    before = (rt.readback(), rt.readback_rgb8())
    rt.render_aov(w, h, 8, seed=4, cameras=cams, projections=LENSES[:2])
    after = (rt.readback(), rt.readback_rgb8())
    assert np.array_equal(before[0][0], after[0][0]) and before[0][1] == after[0][1] and np.array_equal(before[1], after[1])
    rt.render_views_adaptive(cams, w, h, 16, 4, 4, 0.05, seed=4)
    img, st = rt.readback()
    counts, err = rt.readback_adaptive()
    rt.render_aov(w, h, 4, seed=4)
    assert np.array_equal(rt.readback()[0], img) and rt.readback()[1] == st
    c2, e2 = rt.readback_adaptive()
    assert np.array_equal(counts, c2) and np.array_equal(err, e2)
    # accumulation rules: RT_FLAG_ACCUMULATE onto adaptive sums is still refused, onto a fixed render still allowed
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
        rt.render_views(cams, w, h, 4, accumulate=True)
    rt.render(w, h, 4, seed=1)
    rt.render_aov(w, h, 4, seed=2)
    rt.render(w, h, 4, seed=1, sample_begin=4, sample_end=8, accumulate=True)
    ids = rt.primary_ids(w, h)
    rt.render_aov(w, h, 2)
    assert np.array_equal(_ids(rt), ids)


def test_refusals(rt, golden_scene, tmp_path):
    L = gpu.lib()
    sc = golden_scene("tiny")
    with gpu.RtGpu(1, 0) as g:
        p = _abi.rt_render_params(16, 16, 4, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
        assert L.rt_gpu_render_aov(g._h, C.byref(p), None, None) == -4  # RT_ERR_NO_SCENE
        with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
            g.readback_aov()
        g.upload_scene(sc)
        with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
            g.readback_aov()
        g.render(16, 16, 4)
        with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):  # a beauty render is not an AOV render
            g.readback_aov()
        assert L.rt_gpu_render_aov(g._h, None, None, None) == -1

        def bad(**kw):
            q = dict(width=16, height=16, samples=4, sample_begin=0, sample_end=0, mode=_abi.RT_MODE_BEAUTY, seed=0,
                     max_paths_in_flight=0, flags=0, pixel_begin=0, pixel_end=0)
            q.update(kw)
            pp = _abi.rt_render_params(*q.values())
            return L.rt_gpu_render_aov(g._h, C.byref(pp), None, None)

        for kw in (dict(sample_begin=1), dict(sample_end=2), dict(flags=_abi.RT_FLAG_ACCUMULATE), dict(samples=0), dict(width=0),
                   dict(pixel_end=1000), dict(pixel_begin=9, pixel_end=3), dict(mode=7)):
            assert bad(**kw) == -1, kw
        projs = (_abi.rt_projection * 1)(Projection.equirect().to_c())
        assert L.rt_gpu_render_aov(g._h, C.byref(p), None, projs) == -1  # projections without views
        cams = (_abi.rt_camera * 1)(sc.camera().to_c())
        for v in (_abi.rt_views(0, 0, cams), _abi.rt_views(1, 1 << 24, cams)):
            assert L.rt_gpu_render_aov(g._h, C.byref(p), C.byref(v), None) == -1
        cams_nan = (_abi.rt_camera * 1)(sc.camera().to_c())
        cams_nan[0].fov_x = float("nan")
        assert L.rt_gpu_render_aov(g._h, C.byref(p), C.byref(_abi.rt_views(1, 0, cams_nan)), None) == -1
        v1 = _abi.rt_views(1, 0, cams)
        for pj in (_abi.rt_projection(9, 0, 0, 0, 0), _abi.rt_projection(_abi.RT_PROJ_THIN_LENS, -1.0, 1.0, 0, 0),
                   _abi.rt_projection(_abi.RT_PROJ_ORTHOGRAPHIC, 0, 0, 0.0, 1.0)):
            assert L.rt_gpu_render_aov(g._h, C.byref(p), C.byref(v1), C.byref(pj)) == -1
        with pytest.raises(ValueError):
            g.render_aov(16, 16, 4, projections=[Projection.pinhole()])
        # a refused call leaves no AOV render behind
        with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_RENDER"):
            g.readback_aov()
        # a refused call changes nothing: the previous AOV render stays readable
        g.render_aov(16, 16, 2)
        kept = g.readback_aov()
        assert bad(sample_begin=1) == -1
        assert same(kept, g.readback_aov())
    txt = tmp_path / "s.txt"
    txt.write_text("DIMENSIONS 8 8\nRAY_DEPTH 2\nBG_COLOR 0.1 0.2 0.3\nNEW_PRIMITIVE\nBOX 1 2 3\nPOSITION 4 5 6\n")
    from rt_b200 import textscene
    with gpu.RtGpu(1, 0) as g:
        g.upload_text_scene(textscene.load_text_scene(str(txt)))
        with pytest.raises(gpu.RtGpuError, match="RT_ERR_INVALID_ARG"):
            g.render_aov(8, 8, 2)


def test_eight_wide_build_aov():
    """Identity 1, the pixel-centre comparison and the host statement through librt_gpu_wide8.so (k_extend8) in a fresh
    interpreter."""
    if os.environ.get("RT_GPU_LIB"):
        pytest.skip("already the child run")
    lib = os.path.join(ROOT, "raytracing-course-hw-public_b200", "librt_gpu_wide8.so")
    env = dict(os.environ, RT_GPU_LIB=lib)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", "-m", "gpu", os.path.abspath(__file__),
                        "-k", "emission_at_depth_one or pixel_centres or alpha_walk or identities"],
                       env=env, cwd=ROOT, capture_output=True, text=True)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]


def test_wide8_equals_default_library(golden_scene, tmp_path):
    """librt_gpu_wide8.so gives the default library's AOVs on one golden scene (a child process per library)."""
    if os.environ.get("RT_GPU_LIB"):
        pytest.skip("already the child run")
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import rt_b200; from rt_b200 import gpu\n"
            "sc = rt_b200.SceneData.load(%r)\n"
            "with gpu.RtGpu(1, 0) as g:\n"
            "    g.upload_scene(sc); g.render_aov(64, 48, 8, seed=2); a = g.readback_aov()\n"
            "np.savez(sys.argv[1], **a)\n") % (ROOT, os.path.join(ROOT, "tests", "golden", "small_lights.rtsc"))
    out = []
    for lib in ("librt_gpu.so", "librt_gpu_wide8.so"):
        path = str(tmp_path / f"{lib}.npz")
        env = dict(os.environ, RT_GPU_LIB=os.path.join(ROOT, "raytracing-course-hw-public_b200", lib))
        r = subprocess.run([sys.executable, "-c", code, path], env=env, cwd=ROOT, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        out.append(np.load(path))
    a, b = out
    # the two libraries' trees may break a tie differently: the same few-pixel allowance as the path-by-path parity
    close = np.ones(a["depth"].shape, bool)
    for k in NAMES:
        c = np.isclose(a[k], b[k], rtol=1e-4, atol=1e-5)
        close &= c.all(axis=-1) if c.ndim == 3 else c
    print(f"wide8 vs default: {1 - close.mean():.4f} of pixels differ")
    assert close.mean() >= 0.99


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
            g.render_aov(48, 32, 6, seed=5, cameras=cams, projections=LENSES)
            out.append((g.readback_aov(), g.aov_stats()))
    assert same(out[0][0], out[1][0])
    assert out[0][1]["samples"] == out[1][1]["samples"] and out[0][1]["extension_rays"] == out[1][1]["extension_rays"]


def _read_ppm(path):
    data = open(path, "rb").read()
    w, h = (int(x) for x in data.split(b"\n")[1].split())
    return np.frombuffer(data.split(b"\n255\n", 1)[1], np.uint8).reshape(h, w, 3)


def test_python_cli_aov(scene_dir, tmp_path, monkeypatch):
    """RT_AOV: the PFMs decode to readback_aov's arrays of the same camera, projection and seed; the beauty PPM is
    byte-identical to a run without RT_AOV; RT_CAMERAS=all writes <stem>_<i>_<name>.pfm; refusals exit 1."""
    from rt_b200 import cli

    w, h, spp = 64, 48, 8
    src = scene_dir("tiny")
    sc = gltf.load_gltf(src, w / h)
    monkeypatch.setenv("RT_SEED", "5")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "plain.ppm")]) == 0
    monkeypatch.setenv("RT_AOV", "4")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "a.ppm")]) == 0
    assert open(tmp_path / "a.ppm", "rb").read() == open(tmp_path / "plain.ppm", "rb").read()
    monkeypatch.setenv("RT_PROJECTION", "thin_lens:0.05:3")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "t.ppm")]) == 0
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_aov(w, h, 4, seed=5, max_paths_in_flight=128 << 20)
        ref = g.readback_aov()
        g.render_aov(w, h, 4, seed=5, cameras=[sc.camera()], projections=[Projection.thin_lens(0.05, 3.0)], max_paths_in_flight=128 << 20)
        ref_t = {k: v[0] for k, v in g.readback_aov().items()}
    for k in NAMES:
        assert np.array_equal(pfm.read_pfm(tmp_path / f"a_{k}.pfm"), ref[k]), k
        assert np.array_equal(pfm.read_pfm(tmp_path / f"t_{k}.pfm"), ref_t[k]), k
    assert ref["coverage"].max() == 1.0 and not np.array_equal(ref["depth"], ref_t["depth"])
    monkeypatch.delenv("RT_PROJECTION")
    monkeypatch.setenv("RT_CAMERAS", "all")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "v.ppm")]) == 0
    cams = sc.cameras or [sc.camera()]
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_aov(w, h, 4, seed=5, cameras=cams, max_paths_in_flight=128 << 20)
        ref_v = g.readback_aov()
    for i in range(len(cams)):
        for k in NAMES:
            assert np.array_equal(pfm.read_pfm(tmp_path / f"v_{i}_{k}.pfm"), ref_v[k][i]), (i, k)
    monkeypatch.delenv("RT_CAMERAS")
    monkeypatch.setenv("RT_AOV", "4.5")
    assert cli.main(["prog", src, str(w), str(h), str(spp), str(tmp_path / "x.ppm")]) == 1
    assert not (tmp_path / "x.ppm").exists()


def test_cpp_cli_aov(scene_dir, tmp_path):
    exe = os.path.join(ROOT, "bin", "raytracer_b200")
    if not os.path.exists(exe):
        pytest.skip("bin/raytracer_b200 not built (reference headers absent at build time)")
    w, h, spp = 64, 48, 8
    src = scene_dir("tiny")
    env = dict(os.environ, RT_SEED="3")
    assert subprocess.run([exe, src, str(w), str(h), str(spp), str(tmp_path / "p.ppm")], env=env).returncode == 0
    env["RT_AOV"] = "4"
    assert subprocess.run([exe, src, str(w), str(h), str(spp), str(tmp_path / "a.ppm")], env=env).returncode == 0
    assert open(tmp_path / "a.ppm", "rb").read() == open(tmp_path / "p.ppm", "rb").read()
    sc = gltf.load_gltf(src, w / h)
    with gpu.RtGpu(1, 0) as g:
        g.upload_scene(sc)
        g.render_aov(w, h, 4, seed=3, max_paths_in_flight=128 << 20)
        ref = g.readback_aov()
    for k in NAMES:
        assert np.allclose(pfm.read_pfm(tmp_path / f"a_{k}.pfm"), ref[k], rtol=1e-5, atol=1e-6), k
    env["RT_AOV"] = "x"
    assert subprocess.run([exe, src, str(w), str(h), str(spp), str(tmp_path / "x.ppm")], env=env).returncode != 0
