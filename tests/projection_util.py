"""Shared pieces of the projection tests: projected_ray (csrc/projection.cuh) compiled for the host, the device camera
the library makes from an rt_camera, float64 statements of each projection, and a glTF with an orthographic camera."""
import ctypes as C
import json
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "raytracing-course-hw-public_b200", "csrc")

SHIM = r"""
#include <cmath>
#include <cstring>
#include "projection.cuh"
using namespace rt;

// make_camera of rt_gpu.cu: the device camera of an rt_camera (position, right, up, forward, fov_x) for w x h
static Camera mk(const float *s, unsigned w, unsigned h) {
    Camera c;
    c.pos = mk3(s[0], s[1], s[2]);
    c.right = mk3(s[3], s[4], s[5]);
    c.up = mk3(s[6], s[7], s[8]);
    c.fwd = mk3(s[9], s[10], s[11]);
    const float fov_x = s[12];
    c.tan_half_x = std::tan(fov_x / 2);
    const float fov_y = std::atan(std::tan(fov_x / 2) * static_cast<float>(h) / static_cast<float>(w)) * 2;
    c.tan_half_y = std::tan(fov_y / 2);
    c.inv_w2 = 2.0f / static_cast<float>(w);
    c.inv_h2 = 2.0f / static_cast<float>(h);
    return c;
}

extern "C" void make_cam(const float *cam13, unsigned w, unsigned h, float *out16) {
    const Camera c = mk(cam13, w, h);
    std::memcpy(out16, &c, sizeof(Camera));
}

extern "C" void proj_rays(const float *cam13, unsigned w, unsigned h, const void *proj, unsigned n, const float *px, const float *py,
                          const float *lu, const float *lv, float *out) {
    const Camera c = mk(cam13, w, h);
    Projection p;
    std::memcpy(&p, proj, sizeof(Projection));
    for (unsigned i = 0; i < n; ++i) {
        const ProjectedRay r = projected_ray(c, p, px[i], py[i], lu[i], lv[i]);
        const float v[6] = {r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z};
        std::memcpy(out + 6 * i, v, sizeof(v));
    }
}

extern "C" void cam_dirs(const float *cam13, unsigned w, unsigned h, unsigned n, const float *px, const float *py, float *out) {
    const Camera c = mk(cam13, w, h);
    for (unsigned i = 0; i < n; ++i) {
        const f3 d = camera_dir(c, px[i], py[i]);
        out[3 * i] = d.x, out[3 * i + 1] = d.y, out[3 * i + 2] = d.z;
    }
}

extern "C" void discs(unsigned n, const float *lu, const float *lv, float *out) {
    for (unsigned i = 0; i < n; ++i) concentric_disc(lu[i], lv[i], out[2 * i], out[2 * i + 1]);
}
"""


class HostProjection:
    """projected_ray, camera_dir and concentric_disc of projection.cuh, compiled for the host with g++."""

    def __init__(self):
        gxx = shutil.which("g++")
        if not gxx:
            raise RuntimeError("no host C++ compiler")
        self._dir = tempfile.mkdtemp(prefix="rt_projection_")
        src, so = os.path.join(self._dir, "shim.cpp"), os.path.join(self._dir, "libprojection.so")
        with open(src, "w") as f:
            f.write(SHIM)
        subprocess.run([gxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-I" + CSRC, "-I" + os.path.join(ROOT, "include"), "-o", so, src],
                       check=True)
        self.L = C.CDLL(so)

    @staticmethod
    def _cam(cam):
        return np.concatenate([cam.position, cam.right, cam.up, cam.forward, [cam.fov_x]]).astype(np.float32)

    @staticmethod
    def _f(a, n):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float32), (n,)))

    def device_camera(self, cam, w, h):
        """The 16 floats of rt::Camera: pos, right, up, fwd, tan_half_x, tan_half_y, inv_w2, inv_h2."""
        out = np.empty(16, np.float32)
        self.L.make_cam(self._cam(cam).ctypes.data_as(C.c_void_p), w, h, out.ctypes.data_as(C.c_void_p))
        return out

    def rays(self, cam, proj, w, h, px, py, lu=0.5, lv=0.5):
        """[n, 6] float32 (origin, direction) of projected_ray for image points (px, py) and lens samples (lu, lv)."""
        n = len(np.atleast_1d(px))
        args = [self._f(a, n) for a in (px, py, lu, lv)]
        out = np.empty((n, 6), np.float32)
        pc = proj.to_c()
        self.L.proj_rays(self._cam(cam).ctypes.data_as(C.c_void_p), w, h, C.byref(pc), n,
                         *[a.ctypes.data_as(C.c_void_p) for a in args], out.ctypes.data_as(C.c_void_p))
        return out

    def camera_dirs(self, cam, w, h, px, py):
        n = len(np.atleast_1d(px))
        a, b = self._f(px, n), self._f(py, n)
        out = np.empty((n, 3), np.float32)
        self.L.cam_dirs(self._cam(cam).ctypes.data_as(C.c_void_p), w, h, n, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p),
                        out.ctypes.data_as(C.c_void_p))
        return out

    def disc(self, lu, lv):
        n = len(lu)
        a, b = self._f(lu, n), self._f(lv, n)
        out = np.empty((n, 2), np.float32)
        self.L.discs(n, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
        return out


def pixel_centre_rays(hp, cam, proj, w, h):
    """[h * w, 6] rays of the pixel centres through the lens centre, row-major (RT_MODE_PRIMARY_IDS)."""
    y, x = np.divmod(np.arange(w * h), w)
    return hp.rays(cam, proj, w, h, x + np.float32(0.5), y + np.float32(0.5))


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def with_camera_nodes(src, out_name, cameras):
    """The glTF `src` with its camera nodes replaced by `cameras`: a list of (camera dict of the glTF "cameras" array,
    translation) in traversal order, all with the identity rotation."""
    with open(src) as f:
        doc = json.load(f)
    scene = doc["scenes"][doc.get("scene", 0)]
    scene["nodes"] = [i for i in scene["nodes"] if "camera" not in doc["nodes"][i]]
    for cdef, t in cameras:
        doc.setdefault("cameras", []).append(cdef)
        doc["nodes"].append({"camera": len(doc["cameras"]) - 1, "translation": list(map(float, t))})
        scene["nodes"].append(len(doc["nodes"]) - 1)
    out = os.path.join(os.path.dirname(src), out_name)
    with open(out, "w") as f:
        json.dump(doc, f)
    return out
