"""ctypes binding of librt_gpu.so (include/rt_gpu.h) — the CUDA backend. No fallback: a missing library or a
missing GPU raises."""
import ctypes as C
import os

import numpy as np

from . import _abi
from ._abi import (RT_FLAG_ACCUMULATE, RT_MODE_BEAUTY, RT_MODE_PRIMARY_IDS, rt_adaptive_params, rt_camera, rt_geometry_update,
                   rt_projection, rt_render_params, rt_scene_desc, rt_stats, rt_views)

# RT_GPU_LIB selects another build of the same C ABI (kernel A/B experiments, tools/build_variants.sh)
LIB_PATH = os.environ.get("RT_GPU_LIB") or os.path.join(_abi.PKG_DIR, "librt_gpu.so")

# every symbol include/rt_gpu.h declares
SYMBOLS = ["rt_gpu_create", "rt_gpu_destroy", "rt_gpu_upload_scene", "rt_gpu_upload_text_scene", "rt_gpu_render", "rt_gpu_readback",
           "rt_gpu_accum_device_ptr", "rt_gpu_readback_rgb8", "rt_gpu_set_profiling", "rt_gpu_debug_get_bvh", "rt_gpu_fp32_peak", "rt_gpu_last_error",
           "rt_gpu_device_count", "rt_gpu_abi_version", "rt_gpu_render_adaptive", "rt_gpu_readback_adaptive",
           "rt_gpu_render_views", "rt_gpu_render_views_adaptive", "rt_gpu_render_projected", "rt_gpu_update_geometry",
           "rt_gpu_debug_light_pdf"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        L = _abi.load_library(LIB_PATH, "CUDA backend (librt_gpu.so)")
        L.rt_gpu_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
        L.rt_gpu_destroy.argtypes = [C.c_void_p]
        L.rt_gpu_destroy.restype = None
        L.rt_gpu_upload_scene.argtypes = [C.c_void_p, C.POINTER(rt_scene_desc)]
        L.rt_gpu_upload_text_scene.argtypes = [C.c_void_p, C.c_void_p]
        L.rt_gpu_update_geometry.argtypes = [C.c_void_p, C.POINTER(rt_geometry_update)]
        L.rt_gpu_render.argtypes = [C.c_void_p, C.POINTER(rt_render_params)]
        L.rt_gpu_readback.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(rt_stats)]
        L.rt_gpu_render_adaptive.argtypes = [C.c_void_p, C.POINTER(rt_render_params), C.POINTER(rt_adaptive_params)]
        L.rt_gpu_render_views.argtypes = [C.c_void_p, C.POINTER(rt_render_params), C.POINTER(rt_views)]
        L.rt_gpu_render_views_adaptive.argtypes = [C.c_void_p, C.POINTER(rt_render_params), C.POINTER(rt_views),
                                                   C.POINTER(rt_adaptive_params)]
        L.rt_gpu_render_projected.argtypes = [C.c_void_p, C.POINTER(rt_render_params), C.POINTER(rt_views), C.POINTER(rt_projection),
                                              C.POINTER(rt_adaptive_params)]
        L.rt_gpu_readback_adaptive.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rt_gpu_accum_device_ptr.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.rt_gpu_readback_rgb8.argtypes = [C.c_void_p, C.c_void_p]
        L.rt_gpu_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.rt_gpu_debug_get_bvh.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_size_t)]
        L.rt_gpu_fp32_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.rt_gpu_debug_light_pdf.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.rt_gpu_last_error.restype = C.c_char_p
        _lib = L
    return _lib


class RtGpuError(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        msg = lib().rt_gpu_last_error().decode(errors="replace")
        raise RtGpuError(f"{what}: {_abi.STATUS.get(rc, rc)}: {msg}")


def device_count():
    return lib().rt_gpu_device_count()


class RtGpu:
    """One handle = n_gpus devices of this process (rt_gpu_create)."""

    def __init__(self, n_gpus=1, first_device=0):
        self._h = C.c_void_p()
        _check(lib().rt_gpu_create(C.byref(self._h), n_gpus, first_device), "rt_gpu_create")
        self.n_gpus = n_gpus
        self._scene = None
        self._last = None
        self._views = None  # views of the last render when it was render_views: readbacks are [V, H, W, ...]

    def close(self):
        if self._h:
            lib().rt_gpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def upload_scene(self, scene):
        d = scene.desc()
        _check(lib().rt_gpu_upload_scene(self._h, C.byref(d)), "rt_gpu_upload_scene")
        self._scene = scene

    def update_geometry(self, scene):
        """Move the uploaded scene's triangles (rt_gpu_update_geometry): `scene` is a SceneData of the same triangles at
        new positions; its positions, normals, tangents and light_bvh are passed (build the light BVH over the new
        positions with host.build_bvh(tri_pos, select=emissive)).  The library refits its own scene BVH."""
        u = scene.geometry_update()
        _check(lib().rt_gpu_update_geometry(self._h, C.byref(u)), "rt_gpu_update_geometry")

    def upload_text_scene(self, scene):
        """Course text scene (textscene.TextScene); render / readback / primary_ids then work on it."""
        d = scene.desc()
        _check(lib().rt_gpu_upload_text_scene(self._h, C.byref(d)), "rt_gpu_upload_text_scene")
        self._scene = scene

    def set_profiling(self, enable):
        _check(lib().rt_gpu_set_profiling(self._h, int(bool(enable))), "rt_gpu_set_profiling")

    def render(self, width, height, samples, seed=0, sample_begin=0, sample_end=0, mode=RT_MODE_BEAUTY,
               max_paths_in_flight=0, accumulate=False, pixel_begin=0, pixel_end=0):
        p = rt_render_params(width, height, samples, sample_begin, sample_end, mode, seed, max_paths_in_flight,
                             RT_FLAG_ACCUMULATE if accumulate else 0, pixel_begin, pixel_end)
        _check(lib().rt_gpu_render(self._h, C.byref(p)), "rt_gpu_render")
        self._last = (width, height, mode)
        self._views = None

    def render_views(self, cameras, width, height, samples, seed=0, view_base=0, sample_begin=0, sample_end=0,
                     mode=RT_MODE_BEAUTY, max_paths_in_flight=0, accumulate=False, pixel_begin=0, pixel_end=0):
        """Multi-view render (rt_gpu_render_views): every Camera of `cameras` over the uploaded scene in one call, the
        views stacked into one image of W x (V * H) pixels (pixel_begin / pixel_end index it).  Pixel p of view v is
        keyed (view_base + v) * W * H + p, so view v equals a one-view call with view_base = v.  readback() and
        readback_rgb8() then return [V, H, W, 3]."""
        cams = (rt_camera * max(len(cameras), 1))(*[c.to_c() for c in cameras])
        v = rt_views(len(cameras), view_base, cams)
        p = rt_render_params(width, height, samples, sample_begin, sample_end, mode, seed, max_paths_in_flight,
                             RT_FLAG_ACCUMULATE if accumulate else 0, pixel_begin, pixel_end)
        _check(lib().rt_gpu_render_views(self._h, C.byref(p), C.byref(v)), "rt_gpu_render_views")
        self._last = (width, height, mode)
        self._views = len(cameras)

    def _shape(self, *tail):
        w, h, _ = self._last
        return ((self._views,) if self._views is not None else ()) + (h, w) + tail

    def render_adaptive(self, width, height, max_samples, min_samples, step_samples, rel_error, abs_floor=1e-3, seed=0,
                        max_paths_in_flight=0, pixel_begin=0, pixel_end=0):
        """Adaptive render (rt_gpu_render_adaptive): every pixel of the range traces min_samples, then step_samples more
        per round until its relative standard error is <= rel_error or it has max_samples.  readback() then returns
        the per-pixel means, readback_adaptive() the sample counts and errors."""
        p = rt_render_params(width, height, max_samples, 0, 0, RT_MODE_BEAUTY, seed, max_paths_in_flight, 0, pixel_begin,
                             pixel_end)
        a = rt_adaptive_params(min_samples, step_samples, rel_error, abs_floor)
        _check(lib().rt_gpu_render_adaptive(self._h, C.byref(p), C.byref(a)), "rt_gpu_render_adaptive")
        self._last = (width, height, RT_MODE_BEAUTY)
        self._views = None

    def render_views_adaptive(self, cameras, width, height, max_samples, min_samples, step_samples, rel_error, abs_floor=1e-3,
                              seed=0, view_base=0, max_paths_in_flight=0, pixel_begin=0, pixel_end=0):
        """Adaptive multi-view render (rt_gpu_render_views_adaptive): render_adaptive over the stacked image of
        render_views (pixel_begin / pixel_end index it; pixel p of view v is keyed (view_base + v) * W * H + p).
        readback(), readback_rgb8() and readback_adaptive() then return [V, H, W, ...]."""
        cams = (rt_camera * max(len(cameras), 1))(*[c.to_c() for c in cameras])
        v = rt_views(len(cameras), view_base, cams)
        p = rt_render_params(width, height, max_samples, 0, 0, RT_MODE_BEAUTY, seed, max_paths_in_flight, 0, pixel_begin,
                             pixel_end)
        a = rt_adaptive_params(min_samples, step_samples, rel_error, abs_floor)
        _check(lib().rt_gpu_render_views_adaptive(self._h, C.byref(p), C.byref(v), C.byref(a)), "rt_gpu_render_views_adaptive")
        self._last = (width, height, RT_MODE_BEAUTY)
        self._views = len(cameras)

    def render_projected(self, cameras, projections, width, height, samples, seed=0, view_base=0, sample_begin=0, sample_end=0,
                         mode=RT_MODE_BEAUTY, max_paths_in_flight=0, accumulate=False, pixel_begin=0, pixel_end=0, adaptive=None):
        """Projected multi-view render (rt_gpu_render_projected): render_views with projections[v] (a Projection) applied
        to cameras[v].  adaptive=None renders a fixed spp with render_views' contract; adaptive=(min_samples,
        step_samples, rel_error[, abs_floor]) renders with render_views_adaptive's contract, `samples` being the maximum
        spp.  readback(), readback_rgb8() and, when adaptive, readback_adaptive() then return [V, H, W, ...]."""
        if len(projections) != len(cameras):
            raise ValueError(f"render_projected: {len(cameras)} cameras but {len(projections)} projections")
        cams = (rt_camera * max(len(cameras), 1))(*[c.to_c() for c in cameras])
        projs = (rt_projection * max(len(projections), 1))(*[pj.to_c() for pj in projections])
        v = rt_views(len(cameras), view_base, cams)
        p = rt_render_params(width, height, samples, sample_begin, sample_end, mode, seed, max_paths_in_flight,
                             RT_FLAG_ACCUMULATE if accumulate else 0, pixel_begin, pixel_end)
        a = None if adaptive is None else C.byref(rt_adaptive_params(*adaptive) if len(adaptive) == 4 else rt_adaptive_params(*adaptive, 1e-3))
        _check(lib().rt_gpu_render_projected(self._h, C.byref(p), C.byref(v), projs, a), "rt_gpu_render_projected")
        self._last = (width, height, mode)
        self._views = len(cameras)

    def readback_adaptive(self):
        """(sample counts uint32 [H, W], err float32 [H, W]) of the last adaptive render; [V, H, W] each after
        render_views_adaptive."""
        counts = np.empty(self._shape(), np.uint32)
        err = np.empty(self._shape(), np.float32)
        _check(lib().rt_gpu_readback_adaptive(self._h, counts.ctypes.data_as(C.c_void_p), err.ctypes.data_as(C.c_void_p)),
               "rt_gpu_readback_adaptive")
        return counts, err

    def readback(self):
        """(rgb_mean float32 [H, W, 3], or [V, H, W, 3] after render_views / render_views_adaptive; stats dict) of the last beauty render."""
        out = np.empty(self._shape(3), np.float32)
        st = rt_stats()
        _check(lib().rt_gpu_readback(self._h, out.ctypes.data_as(C.c_void_p), None, C.byref(st)), "rt_gpu_readback")
        return out, st.as_dict()

    def readback_into(self, out):
        """Readback into a caller-provided (e.g. pinned) float32 array of W*H*3 elements."""
        st = rt_stats()
        _check(lib().rt_gpu_readback(self._h, C.c_void_p(out.ctypes.data), None, C.byref(st)), "rt_gpu_readback")
        return st.as_dict()

    def stats(self):
        st = rt_stats()
        _check(lib().rt_gpu_readback(self._h, None, None, C.byref(st)), "rt_gpu_readback")
        return st.as_dict()

    def readback_rgb8(self):
        out = np.empty(self._shape(3), np.uint8)
        _check(lib().rt_gpu_readback_rgb8(self._h, out.ctypes.data_as(C.c_void_p)), "rt_gpu_readback_rgb8")
        return out

    def primary_ids(self, width, height, cameras=None, view_base=0, projections=None):
        """Primary-hit ids [H, W] of the scene's camera, or [V, H, W] of `cameras` (render_views; render_projected with
        `projections`)."""
        if cameras is None:
            self.render(width, height, 1, mode=RT_MODE_PRIMARY_IDS)
        elif projections is not None:
            self.render_projected(cameras, projections, width, height, 1, view_base=view_base, mode=RT_MODE_PRIMARY_IDS)
        else:
            self.render_views(cameras, width, height, 1, view_base=view_base, mode=RT_MODE_PRIMARY_IDS)
        ids = np.empty(self._shape(), np.int32)
        _check(lib().rt_gpu_readback(self._h, None, ids.ctypes.data_as(C.c_void_p), None), "rt_gpu_readback")
        return ids

    def debug_bvh(self, which, dtype):
        """Diagnostic download of the device-built scene BVH (rt_gpu_debug_get_bvh); numpy array of `dtype`."""
        n = C.c_size_t(0)
        _check(lib().rt_gpu_debug_get_bvh(self._h, which, None, C.byref(n)), "rt_gpu_debug_get_bvh")
        out = np.zeros(n.value // np.dtype(dtype).itemsize, dtype)
        if n.value:
            _check(lib().rt_gpu_debug_get_bvh(self._h, which, out.ctypes.data_as(C.c_void_p), C.byref(n)), "rt_gpu_debug_get_bvh")
        return out

    def debug_light_pdf(self, rays):
        """Diagnostic: the light pdf the next k_shade would read for each of `rays` (n x 6 float32: origin, direction) as a
        pending ray (rt_gpu_debug_light_pdf); float32 [n]."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        out = np.zeros(len(rays), np.float32)
        _check(lib().rt_gpu_debug_light_pdf(self._h, len(rays), rays.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)),
               "rt_gpu_debug_light_pdf")
        return out

    def fp32_peak_tflops(self):
        v = C.c_double()
        _check(lib().rt_gpu_fp32_peak(self._h, C.byref(v)), "rt_gpu_fp32_peak")
        return v.value

    def accum_device_ptr(self):
        """(device pointer, n_floats) of device 0's float4 per-pixel sums (for an external collective)."""
        p = C.c_void_p()
        n = C.c_size_t()
        _check(lib().rt_gpu_accum_device_ptr(self._h, C.byref(p), C.byref(n)), "rt_gpu_accum_device_ptr")
        return p.value, n.value
