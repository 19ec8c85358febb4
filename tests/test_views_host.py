"""Multi-view rendering without a GPU: the stacked-pixel split of csrc/views.cuh compiled for the host (the function
k_generate_views evaluates), the new C ABI symbol and struct, the no-device failure, and the glTF loader's list of
every camera node."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from views_scene import with_three_cameras, without_cameras

import rt_b200  # noqa: F401
from rt_b200 import _abi, gltf, gpu

CSRC = os.path.join(ROOT, "raytracing-course-hw-public_b200", "csrc")

SHIM = r"""
#include "views.cuh"
extern "C" void split_many(const unsigned *pixel, unsigned n, unsigned width, unsigned height, unsigned *out) {
    for (unsigned i = 0; i < n; ++i) {
        const rt::ViewPixel v = rt::split_view_pixel(pixel[i], width, height);
        out[3 * i] = v.view;
        out[3 * i + 1] = v.x;
        out[3 * i + 2] = v.y;
    }
}
"""


@pytest.fixture(scope="module")
def split(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no host C++ compiler")
    d = tmp_path_factory.mktemp("views_split")
    src, so = d / "shim.cpp", d / "libviews_split.so"
    src.write_text(SHIM)
    subprocess.run([gxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-I" + CSRC, "-o", str(so), str(src)], check=True)
    L = C.CDLL(str(so))
    L.split_many.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_void_p]
    L.split_many.restype = None

    def run(pixels, w, h):
        p = np.ascontiguousarray(pixels, np.uint32)
        out = np.empty((len(p), 3), np.uint32)
        L.split_many(p.ctypes.data, len(p), w, h, out.ctypes.data)
        return out

    return run


def expect(pixels, w, h):
    view, local = np.divmod(np.asarray(pixels, np.int64), w * h)
    y, x = np.divmod(local, w)
    return np.stack([view, x, y], 1)


@pytest.mark.parametrize("w,h,v", [(1, 1, 5), (8, 4, 3), (7, 5, 4), (96, 64, 5), (1000, 1000, 4), (3, 1, 9)])
def test_split_matches_divmod(split, w, h, v):
    pixels = np.arange(w * h * v, dtype=np.int64)
    if len(pixels) > 200_000:
        pixels = np.unique(np.concatenate([pixels[:5000], pixels[-5000:], np.random.default_rng(1).integers(0, len(pixels), 50_000)]))
    assert np.array_equal(split(pixels, w, h), expect(pixels, w, h))


@pytest.mark.parametrize("w,h", [(65536, 32768), (46341, 46341), (1920, 1080), (4096, 4093)])
def test_split_near_the_top_of_the_key_range(split, w, h):
    """Stacked pixels (and keys) up to 2^32 - 1: the largest view count with V * W * H <= 2^32."""
    v = (1 << 32) // (w * h)
    top = v * w * h
    pixels = np.unique(np.concatenate([np.arange(max(top - 4096, 0), top), np.arange(0, 4096),
                                       np.random.default_rng(2).integers(0, top, 20_000)]))
    assert pixels.max() <= 0xFFFFFFFF
    assert np.array_equal(split(pixels, w, h), expect(pixels, w, h))


def test_views_symbol_and_struct():
    assert "rt_gpu_render_views" in gpu.SYMBOLS
    getattr(C.CDLL(gpu.LIB_PATH), "rt_gpu_render_views")
    assert C.sizeof(_abi.rt_views) == 16
    assert C.sizeof(_abi.rt_camera) == 52 and C.sizeof(_abi.rt_render_params) == 48  # unchanged
    assert _abi.RT_GPU_ABI_VERSION == 1


def test_render_views_fails_without_a_device():
    """In a child process that sees no device (so that this runs on a GPU machine as well)."""
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import gpu\n"
            "cam = rt_b200.Camera([0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, -1], 1.0)\n"
            "try:\n    gpu.RtGpu(1, 0).render_views([cam, cam], 8, 8, 4)\n"
            "except gpu.RtGpuError as e:\n    print(e)\n    sys.exit(0)\nsys.exit(1)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "RT_ERR_NO_DEVICE" in r.stdout, r.stdout + r.stderr


def test_camera_round_trip():
    cam = rt_b200.Camera([1, 2, 3], [1, 0, 0], [0, 1, 0], [0, 0, -1], 0.75)
    c = cam.to_c()
    assert list(c.position) == [1, 2, 3] and list(c.forward) == [0, 0, -1] and c.fov_x == np.float32(0.75)
    assert cam == rt_b200.Camera(c.position, c.right, c.up, c.forward, c.fov_x)
    assert cam != rt_b200.Camera([1, 2, 3], [1, 0, 0], [0, 1, 0], [0, 0, -1], np.nextafter(np.float32(0.75), np.float32(1)))


def test_gltf_returns_every_camera(scene_dir):
    src = scene_dir("tiny")
    path = with_three_cameras(src, "tiny_three_cameras.gltf")
    one = gltf.load_gltf(src, 64 / 48)
    three = gltf.load_gltf(path, 64 / 48)
    assert len(one.cameras) == 1 and one.cameras[0] == one.camera()
    assert len(three.cameras) == 3
    own = one.camera()
    # traversal order: the moved copy (0.4 along x, same axes), the narrower higher one, the scene's own camera
    assert np.array_equal(three.cameras[0].position, own.position + np.float32([0.4, 0, 0]))
    assert np.array_equal(three.cameras[0].forward, own.forward) and three.cameras[0].fov_x == own.fov_x
    assert three.cameras[1].position[1] > own.position[1] and three.cameras[1].fov_x < own.fov_x
    assert three.cameras[2] == own
    # the scene camera is the last camera node, bit for bit, and the scene's arrays are those of the one-camera file
    assert three.camera() == three.cameras[-1]
    for k in ("tri_pos", "tri_normals", "tri_uv", "tri_tangents", "tri_material", "materials", "textures", "texels"):
        assert np.array_equal(getattr(three, k), getattr(one, k)), k
    assert np.array_equal(three.scene_bvh.nodes, one.scene_bvh.nodes) and np.array_equal(three.light_bvh.objects, one.light_bvh.objects)


def test_gltf_without_cameras_has_none(scene_dir):
    s = gltf.load_gltf(without_cameras(scene_dir("tiny"), "tiny_no_camera.gltf"), 1.0)
    assert s.cameras == []
    assert s.camera() == rt_b200.Camera([0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0], 0.0)  # Camera{} defaults
