"""AOV render (rt_gpu_render_aov) without a GPU: hc_aov, the host compilation of aov_visit over the camera rays and traversal
of hc_render, against the reference's pinned pixel-centre hit data; alpha coverage against its binomial expectation;
the refusals that need no device; the PFM writer and the CLI's RT_AOV refusals."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, golden_array

from rt_b200 import _abi, cli, gpu, pfm

SCENES = ["tiny", "small_lights", "texmaps", "texall", "tiny_lt", "small_lights_lt"]  # the scenes with pinned hit data


@pytest.fixture(scope="module")
def hc():
    L = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libaovcheck.so"))  # libhostcheck.so + hc_aov
    L.hc_aov.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, C.c_void_p]
    L.hc_hitinfo.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    return L


def hc_aov(hc, scene, w, h, samples, seed=0, centre=False):
    """{albedo, normal, emission: [H, W, 3], depth, coverage: [H, W]} of the host statement"""
    d = scene.desc()
    out = np.zeros((h, w, 11), np.float32)
    assert hc.hc_aov(C.byref(d), w, h, samples, seed, int(centre), out.ctypes.data_as(C.c_void_p)) == 0
    return {"albedo": out[..., 0:3], "normal": out[..., 3:6], "emission": out[..., 6:9], "depth": out[..., 9], "coverage": out[..., 10]}


def hitinfo(hc, scene, w, h):
    d = scene.desc()
    info = np.zeros((h, w, 18), np.float32)
    assert hc.hc_hitinfo(C.byref(d), w, h, info.ctypes.data_as(C.c_void_p)) == 0
    return info


@pytest.mark.parametrize("name", SCENES)
def test_pixel_centres_are_the_reference_hit_data(name, hc, manifest, golden_scene):
    """centre=True: on pixels whose first hit has alpha 1 the AOVs are make_surface's values of the reference's pinned
    pixel-centre hits (the host's own hit data bit for bit, the reference's within test_device_hit_data_matches_reference's
    tolerances); coverage is ids >= 0 there and 0 on misses."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    a = hc_aov(hc, sc, w, h, 1, centre=True)
    info = hitinfo(hc, sc, w, h)
    ref = golden_array(f"{name}_hitinfo.f32", np.float32, (h, w, 18))
    ids = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    opaque = (ids >= 0) & (ref[..., 10] == 1.0) & (info[..., 10] == 1.0)
    assert opaque.sum() > 0.2 * w * h
    got = np.concatenate([a["depth"][..., None], a["normal"], a["albedo"], a["emission"]], axis=2)[opaque]
    cols = np.r_[0, 4:7, 7:10, 11:14]
    assert np.array_equal(got, info[opaque][:, cols])
    diff = np.abs(got - ref[opaque][:, cols])
    diff[:, 0] /= np.maximum(ref[opaque][:, 0], 1.0)  # t relative
    assert np.quantile(diff, 0.999) < 1e-4 and diff.max() < 5e-3
    assert np.array_equal(a["coverage"][opaque], np.ones(opaque.sum(), np.float32))
    miss = ids < 0
    assert np.all(a["coverage"][miss] == 0) and np.all(a["depth"][miss] == 0) and np.all(a["albedo"][miss] == 0)


def test_alpha_coverage_converges_to_alpha(hc, golden_scene):
    """texall at ray depth 1 (no surface behind a pass-through counts): the coverage of a pixel whose every hit is one
    surface of alpha a is a binomial mean of the beauty path's alpha coins, within 5 standard deviations of a."""
    sc = copy.copy(golden_scene("texall"))
    sc.ray_depth = 1
    w, h, spp, sub = 40, 32, 1024, 4
    a = hc_aov(hc, sc, w, h, spp, seed=11)
    # alpha at sub x sub points spread over each pixel: a pixel qualifies when every point hits with the same alpha
    fine = hitinfo(hc, sc, w * sub, h * sub).reshape(h, sub, w, sub, 18).transpose(0, 2, 1, 3, 4).reshape(h, w, sub * sub, 18)
    hit_all = np.all(fine[..., 0] > 0, axis=2)
    alpha = fine[..., 10]
    same = hit_all & np.all(alpha == alpha[..., :1], axis=2)
    partial = same & (alpha[..., 0] > 0.02) & (alpha[..., 0] < 0.98)
    assert partial.sum() >= 20, partial.sum()
    p = alpha[..., 0][partial].astype(np.float64)
    cov = a["coverage"][partial].astype(np.float64)
    bound = 5.0 * np.sqrt(p * (1 - p) / spp)
    assert np.all(np.abs(cov - p) <= bound), np.max(np.abs(cov - p) / bound)


def test_ray_depth_zero_gives_zeros(hc, golden_scene):
    sc = copy.copy(golden_scene("tiny"))
    sc.ray_depth = 0
    a = hc_aov(hc, sc, 16, 12, 4)
    assert all(np.all(v == 0) for v in a.values())


def test_symbols_and_null_handle():
    """The entry points exist in both libraries; a null handle or null params are refused without a device."""
    L = gpu.lib()
    assert "rt_gpu_render_aov" in gpu.SYMBOLS and "rt_gpu_readback_aov" in gpu.SYMBOLS
    for lib in ("librt_gpu.so", "librt_gpu_wide8.so"):
        so = C.CDLL(os.path.join(ROOT, "raytracing-course-hw-public_b200", lib))
        so.rt_gpu_render_aov, so.rt_gpu_readback_aov
    p = _abi.rt_render_params(16, 16, 4, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
    assert L.rt_gpu_render_aov(None, C.byref(p), None, None) == -1  # RT_ERR_INVALID_ARG
    assert L.rt_gpu_readback_aov(None, None, None, None, None, None, None) == -1
    header = open(os.path.join(ROOT, "include", "rt_gpu.h")).read()
    assert "int rt_gpu_render_aov(" in header and "int rt_gpu_readback_aov(" in header


def test_pfm_round_trip(tmp_path):
    rng = np.random.default_rng(3)
    rgb = rng.normal(size=(5, 7, 3)).astype(np.float32)
    one = rng.normal(size=(5, 7)).astype(np.float32)
    pfm.write_pfm(tmp_path / "a.pfm", rgb)
    pfm.write_pfm(tmp_path / "b.pfm", one)
    raw = open(tmp_path / "a.pfm", "rb").read()
    assert raw.startswith(b"PF\n7 5\n-1\n") and len(raw) == len(b"PF\n7 5\n-1\n") + rgb.nbytes
    # rows bottom to top: the file's first row is the image's last
    assert np.array_equal(np.frombuffer(raw[len(b"PF\n7 5\n-1\n"):][:7 * 12], "<f4").reshape(7, 3), rgb[-1])
    assert open(tmp_path / "b.pfm", "rb").read().startswith(b"Pf\n7 5\n-1\n")
    assert np.array_equal(pfm.read_pfm(tmp_path / "a.pfm"), rgb) and np.array_equal(pfm.read_pfm(tmp_path / "b.pfm"), one)
    with pytest.raises(ValueError):
        pfm.write_pfm(tmp_path / "c.pfm", np.zeros((2, 2, 2), np.float32))


def test_parse_aov():
    assert cli.parse_aov(None) == 0 and cli.parse_aov("") == 0 and cli.parse_aov("0") == 0 and cli.parse_aov("16") == 16
    for bad in ("-1", "1.5", "x", " 4"):
        with pytest.raises(ValueError):
            cli.parse_aov(bad)
    assert cli.aov_paths("out/img.ppm", "_2")["depth"] == "out/img_2_depth.pfm"


def test_cli_refusals(scene_dir, tmp_path, monkeypatch):
    """Malformed RT_AOV, RT_AOV with a text scene and RT_AOV with RT_FRAMES exit 1 before any render."""
    src = scene_dir("tiny")
    monkeypatch.setenv("RT_AOV", "many")
    assert cli.main(["prog", src, "16", "16", "4", str(tmp_path / "a.ppm")]) == 1
    txt = tmp_path / "s.txt"
    txt.write_text("DIMENSIONS 8 8\nRAY_DEPTH 2\nBG_COLOR 0.1 0.2 0.3\n")
    monkeypatch.setenv("RT_AOV", "4")
    assert cli.main(["prog", str(txt), "8", "8", "4", str(tmp_path / "t.ppm")]) == 1
    monkeypatch.setenv("RT_FRAMES", "2:24")
    assert cli.main(["prog", src, "16", "16", "4", str(tmp_path / "f.ppm")]) == 1
    assert not any(tmp_path.glob("*.p?m"))
