"""Camera projections without a GPU: projected_ray of csrc/projection.cuh compiled for the host against a float64
statement of each projection, the uniformity of the lens sampling, the new C ABI symbol and struct, the argument and
no-device failures, and the glTF loader's orthographic camera nodes."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy import stats

from conftest import ROOT
from projection_util import HostProjection, unit, with_camera_nodes

import rt_b200
from rt_b200 import _abi, gltf, gpu
from rt_b200._abi import Projection

NAME = "rt_gpu_render_projected"


@pytest.fixture(scope="module")
def hp():
    try:
        return HostProjection()
    except RuntimeError as e:
        pytest.skip(str(e))


def random_cameras(seed, n=6):
    """(camera, W, H) with random orthonormal bases (glTF convention: right x up = -forward), positions and fields of view."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        right, up = q[:, 0], q[:, 1]
        fwd = -np.cross(right, up)
        w, h = int(rng.integers(1, 400)), int(rng.integers(1, 300))
        cam = rt_b200.Camera(rng.uniform(-50, 50, 3), right, up, fwd, rng.uniform(0.2, 2.5))
        out.append((cam, w, h))
    return out


def points(seed, w, h, n=4000):
    rng = np.random.default_rng(seed)
    px = (rng.integers(0, w, n) + rng.random(n)).astype(np.float32)
    py = (rng.integers(0, h, n) + rng.random(n)).astype(np.float32)
    return px, py, rng.random(n).astype(np.float32), rng.random(n).astype(np.float32)


def basis(hp, cam, w, h):
    c = hp.device_camera(cam, w, h).astype(np.float64)
    return c[0:3], c[3:6], c[6:9], c[9:12], c[12], c[13], c[14], c[15]


@pytest.mark.parametrize("seed", range(4))
def test_pinhole_is_camera_dir_bit_for_bit(hp, seed):
    for cam, w, h in random_cameras(seed):
        px, py, lu, lv = points(seed, w, h)
        r = hp.rays(cam, Projection.pinhole(), w, h, px, py, lu, lv)
        assert np.array_equal(r[:, 3:].view(np.uint32), hp.camera_dirs(cam, w, h, px, py).view(np.uint32))
        assert np.array_equal(r[:, :3], np.broadcast_to(cam.position, (len(px), 3)))
        # a thin lens without aperture, and one sampled at the lens centre, is the pinhole
        for proj, a, b in ((Projection.thin_lens(0.0, 3.0), lu, lv), (Projection.thin_lens(0.0, 0.0), lu, lv),
                           (Projection.thin_lens(0.7, 3.0), 0.5, 0.5)):
            assert np.array_equal(hp.rays(cam, proj, w, h, px, py, a, b).view(np.uint32), r.view(np.uint32)), proj


@pytest.mark.parametrize("seed", range(4))
def test_thin_lens_against_float64(hp, seed):
    for cam, w, h in random_cameras(seed):
        px, py, lu, lv = points(seed, w, h)
        ap, focus = np.float32(0.05 + seed * 0.3), np.float32(1.5 + seed * 4)
        r = hp.rays(cam, Projection.thin_lens(ap, focus), w, h, px, py, lu, lv).astype(np.float64)
        pos, right, up, fwd, tx, ty, iw, ih = basis(hp, cam, w, h)
        a, b = (px * iw - 1) * tx, (py * ih - 1) * ty
        d = unit(a[:, None] * right - b[:, None] * up + fwd)
        focus_pt = pos + d * (float(focus) / (d @ fwd))[:, None]
        # concentric map, float64
        x, y = 2 * lu.astype(np.float64) - 1, 2 * lv.astype(np.float64) - 1
        big = np.abs(x) > np.abs(y)
        rad = np.where(big, x, y)
        with np.errstate(divide="ignore", invalid="ignore"):
            phi = np.where(big, np.pi / 4 * (y / x), np.pi / 2 - np.pi / 4 * (x / y))
        lens = pos + (float(ap) * rad * np.cos(phi))[:, None] * right + (float(ap) * rad * np.sin(phi))[:, None] * up
        scale = np.abs(pos).max() + 1
        assert np.abs(r[:, :3] - lens).max() <= 4e-6 * scale
        assert np.abs(r[:, 3:] - unit(focus_pt - lens)).max() <= 2e-5
        # every ray of a pixel point passes through its focus point: the plane at focus_distance is sharp
        t = ((focus_pt - r[:, :3]) * r[:, 3:]).sum(1)
        miss = np.linalg.norm(r[:, :3] + t[:, None] * r[:, 3:] - focus_pt, axis=1)
        assert miss.max() <= 2e-5 * (scale + float(focus) / np.abs(d @ fwd).min())


@pytest.mark.parametrize("seed", range(4))
def test_orthographic_against_float64(hp, seed):
    for cam, w, h in random_cameras(seed):
        px, py, lu, lv = points(seed, w, h)
        hw, hh = np.float32(0.3 + seed), np.float32(0.2 + 2 * seed)
        r = hp.rays(cam, Projection.orthographic(hw, hh), w, h, px, py, lu, lv)
        fwd32 = np.asarray(cam.forward, np.float32)
        expect_d = hp.rays(cam, Projection.orthographic(hw, hh), w, h, np.float32([0.5]), np.float32([0.5]))[0, 3:]
        assert (r[:, 3:] == expect_d).all(), "every orthographic direction is normalize(forward)"
        assert np.abs(expect_d - fwd32).max() <= 1e-6
        pos, right, up, fwd, tx, ty, iw, ih = basis(hp, cam, w, h)
        a, b = (px * iw - 1) * float(hw), (py * ih - 1) * float(hh)
        o = pos + a[:, None] * right - b[:, None] * up
        assert np.abs(r[:, :3].astype(np.float64) - o).max() <= 4e-6 * (np.abs(pos).max() + hw + hh)
        # the corners of the image span [-half_width, half_width] x [-half_height, half_height] in the camera plane
        c = hp.rays(cam, Projection.orthographic(hw, hh), w, h, np.float32([0, w]), np.float32([0, h]))[:, :3].astype(np.float64)
        np.testing.assert_allclose((c - pos) @ right, [-hw, hw], atol=1e-4 * (np.abs(pos).max() + hw))
        np.testing.assert_allclose((c - pos) @ up, [hh, -hh], atol=1e-4 * (np.abs(pos).max() + hh))


def test_orthographic_axis_aligned_has_no_zero_component(hp):
    """A zero direction component turns the node slab tests into NaN (no culling on that axis): an axis-aligned
    orthographic view gets +-2^-80 instead, and is otherwise forward."""
    cam = rt_b200.Camera([1, 2, 3], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)
    px, py, lu, lv = points(0, 64, 48)
    d = hp.rays(cam, Projection.orthographic(2, 1.5), 64, 48, px, py, lu, lv)[:, 3:]
    assert (d != 0).all() and (np.abs(d[:, :2]) == np.float32(2.0 ** -80)).all() and (d[:, 2] == -1).all()


@pytest.mark.parametrize("seed", range(4))
def test_equirect_against_float64(hp, seed):
    for cam, w, h in random_cameras(seed):
        px, py, lu, lv = points(seed, w, h)
        r = hp.rays(cam, Projection.equirect(), w, h, px, py, lu, lv).astype(np.float64)
        assert np.array_equal(r[:, :3], np.broadcast_to(cam.position, (len(px), 3)))
        d = r[:, 3:]
        assert np.abs(np.linalg.norm(d, axis=1) - 1).max() <= 2e-7
        pos, right, up, fwd = basis(hp, cam, w, h)[:4]
        u, v = (px - 0.5) / w, (py - 0.5) / h
        phi, theta = (u - 0.5) * 2 * np.pi, (0.5 - v) * np.pi
        expect = (np.cos(theta) * np.sin(phi))[:, None] * right + np.sin(theta)[:, None] * up + (np.cos(theta) * np.cos(phi))[:, None] * fwd
        assert np.abs(d - expect).max() <= 2e-5 * max(w, h) / 64 + 2e-6
        # the stated angles: theta from the up component, phi from the right / forward components
        np.testing.assert_allclose(d @ up, np.sin(theta), atol=2e-6)
        ok = np.cos(theta) > 1e-2
        dphi = np.angle(np.exp(1j * (np.arctan2(d @ right, d @ fwd) - phi)))[ok]
        assert np.abs(dphi).max() <= 1e-3


def test_equirect_follows_bg_at(hp):
    """With forward = +x, right = +z, up = +y the centre of pixel (i, j) looks up texel (i, j) of a map of the view's size
    in bg_at's coordinates x = 0.5 + 0.5 atan2(d.z, d.x) / pi, y = 0.5 - asin(d.y) / pi (texel i at x = i / W)."""
    w, h = 64, 32
    cam = rt_b200.Camera([0, 0, 0], [0, 0, 1], [0, 1, 0], [1, 0, 0], 1.0)
    y, x = np.divmod(np.arange(w * h), w)
    d = hp.rays(cam, Projection.equirect(), w, h, x + np.float32(0.5), y + np.float32(0.5))[:, 3:].astype(np.float64)
    tx = (0.5 + 0.5 * np.arctan2(d[:, 2], d[:, 0]) / np.pi) * w
    ty = (0.5 - np.arcsin(np.clip(d[:, 1], -1, 1)) / np.pi) * h
    off_pole = y > 0  # row 0 looks straight up, where every x names the same direction
    assert np.abs(np.angle(np.exp(2j * np.pi * (tx - x) / w)))[off_pole].max() * w / (2 * np.pi) <= 1e-3
    assert np.abs(ty - y).max() <= 1e-3


def test_concentric_disc_is_uniform(hp):
    """A seeded jittered grid of (lu, lv) maps into the unit disc; its counts in 8 rings x 16 sectors of equal area pass
    a chi-square test (and (0.5, 0.5) is the centre)."""
    n = 512
    rng = np.random.default_rng(11)
    g = (np.arange(n)[:, None] + rng.random((n, n))) / n
    lu = g.reshape(-1).astype(np.float32)
    lv = ((np.arange(n)[None, :] + rng.random((n, n))) / n).reshape(-1).astype(np.float32)
    p = hp.disc(lu, lv).astype(np.float64)
    r2 = (p ** 2).sum(1)
    assert r2.max() <= 1 + 1e-6
    ring = np.minimum((r2 * 8).astype(int), 7)
    sector = ((np.arctan2(p[:, 1], p[:, 0]) + np.pi) / (2 * np.pi) * 16).astype(int) % 16
    counts = np.bincount(ring * 16 + sector, minlength=128)
    chi2, pval = stats.chisquare(counts)
    assert pval > 1e-3, (chi2, pval, counts)
    assert np.array_equal(hp.disc(np.float32([0.5]), np.float32([0.5])), np.zeros((1, 2), np.float32))


def test_symbol_is_exported_and_declared():
    assert NAME in gpu.SYMBOLS
    getattr(C.CDLL(gpu.LIB_PATH), NAME)
    with open(os.path.join(ROOT, "include", "rt_gpu.h")) as f:
        text = f.read()
    assert f"int {NAME}(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views," in text
    for k, v in (("PINHOLE", 0), ("THIN_LENS", 1), ("ORTHOGRAPHIC", 2), ("EQUIRECT", 3)):
        assert f"#define RT_PROJ_{k} {v}u" in text
        assert getattr(_abi, f"RT_PROJ_{k}") == v


def test_struct_sizes_are_unchanged():
    assert C.sizeof(_abi.rt_projection) == 20
    assert C.sizeof(_abi.rt_views) == 16 and C.sizeof(_abi.rt_adaptive_params) == 16
    assert C.sizeof(_abi.rt_camera) == 52 and C.sizeof(_abi.rt_render_params) == 48
    assert C.sizeof(_abi.rt_stats) == 120
    assert _abi.RT_GPU_ABI_VERSION == 1


def test_null_arguments_are_refused_before_any_device_work():
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    cams = (_abi.rt_camera * 1)(rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0).to_c())
    projs = (_abi.rt_projection * 1)(Projection.equirect().to_c())
    p = _abi.rt_render_params(8, 8, 16, 0, 0, _abi.RT_MODE_BEAUTY, 0, 0, 0, 0, 0)
    v = _abi.rt_views(1, 0, cams)
    assert L.rt_gpu_render_projected(None, C.byref(p), C.byref(v), projs, None) == bad
    assert L.rt_gpu_render_projected(None, None, None, None, None) == bad
    assert NAME in L.rt_gpu_last_error().decode()


def test_projection_parse_and_equality():
    assert Projection.parse("thin_lens:0.25:3.5") == Projection.thin_lens(0.25, 3.5)
    assert Projection.parse("ortho:2:1.5") == Projection.orthographic(2, 1.5)
    assert Projection.parse("equirect") == Projection.equirect() and Projection.parse("pinhole") == Projection()
    assert Projection.thin_lens(0.25, 3.5) != Projection.thin_lens(0.25, np.nextafter(np.float32(3.5), np.float32(4)))
    for bad in ("fisheye", "ortho:1", "thin_lens:1:2:3", "equirect:1", "ortho:a:b"):
        with pytest.raises(ValueError):
            Projection.parse(bad)
    c = Projection.orthographic(2, 1.5).to_c()
    assert (c.kind, c.half_width, c.half_height, c.aperture_radius) == (_abi.RT_PROJ_ORTHOGRAPHIC, 2.0, 1.5, 0.0)


@pytest.mark.parametrize("via", ["python", "c"])
def test_fails_without_a_device(via):
    """In a child process that sees no device: the Python method raises RT_ERR_NO_DEVICE, and so does the C sequence up
    to the call."""
    if via == "python":
        code = ("import sys; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import gpu\n"
                "cam = rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)\n"
                "pj = [rt_b200.Projection.thin_lens(0.1, 2.0), rt_b200.Projection.equirect()]\n"
                "try:\n    gpu.RtGpu(1, 0).render_projected([cam, cam], pj, 8, 8, 16)\n"
                "except gpu.RtGpuError as e:\n    print(e)\n    sys.exit(0)\nsys.exit(1)\n")
    else:
        code = ("import sys, ctypes as C; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import _abi, gpu\n"
                "L = gpu.lib(); h = C.c_void_p()\n"
                "rc = L.rt_gpu_create(C.byref(h), 1, 0)\n"
                "if rc == 0:\n    sys.exit(1)\n"
                "print(_abi.STATUS[rc], L.rt_gpu_last_error().decode())\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "RT_ERR_NO_DEVICE" in r.stdout, r.stdout + r.stderr


def test_gltf_orthographic_camera(scene_dir):
    """An orthographic camera node joins SceneData.cameras with its xmag / ymag; perspective entries and the scene camera
    (the last perspective node) are those of a file without it, bit for bit."""
    src = scene_dir("tiny")
    base = gltf.load_gltf(src, 64 / 48)
    own = base.cameras[-1]
    with open(src) as f:
        import json
        doc = json.load(f)
    persp = doc["cameras"][next(n for n in doc["nodes"] if "camera" in n)["camera"]]
    t = [float(x) for x in own.position]
    ortho = {"type": "orthographic", "orthographic": {"xmag": 1.25, "ymag": 0.75, "znear": 0.01, "zfar": 100.0}}
    only_persp = gltf.load_gltf(with_camera_nodes(src, "tiny_persp.gltf", [(persp, t)]), 64 / 48)
    mixed = gltf.load_gltf(with_camera_nodes(src, "tiny_ortho.gltf", [(persp, t), (ortho, [0.5, 1.0, 4.0])]), 64 / 48)
    assert len(mixed.cameras) == len(mixed.projections) == 2
    assert mixed.cameras[0] == only_persp.cameras[0] and mixed.projections[0] == Projection.pinhole()
    assert mixed.projections[1] == Projection.orthographic(1.25, 0.75)
    o = mixed.cameras[1]
    assert np.array_equal(o.position, np.float32([0.5, 1.0, 4.0]))
    assert np.array_equal(o.right, [1, 0, 0]) and np.array_equal(o.up, [0, 1, 0]) and np.array_equal(o.forward, [0, 0, -1])
    # the scene camera stays the last perspective node
    assert mixed.camera() == only_persp.camera() == only_persp.cameras[-1]
    for k in ("tri_pos", "tri_normals", "tri_material"):
        assert np.array_equal(getattr(mixed, k), getattr(base, k)), k
    # a file of perspective cameras only: one pinhole projection per camera
    assert base.projections == [Projection.pinhole()] * len(base.cameras)
