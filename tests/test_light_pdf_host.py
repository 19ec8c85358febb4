"""Light pdfs of the host compilation of the device math (hc_light_pdf: light_pdf over the exact binary light nodes, and
light_pdf_q8 over the 8-wide quantised ones, the scene packed as hc_render packs it) against the float64 brute force
hc_brute_light_pdf, on the scenarios of light_scenarios.py.  No GPU needed.  Also the numpy statement of the reference
against the C++ one, and the refusals of rt_gpu_debug_light_pdf that come before any device work."""
import ctypes as C
import os

import numpy as np
import pytest

import hit_scenarios as hs
import light_scenarios as ls
from rt_b200 import _abi, gltf, gpu

from conftest import ROOT

NAME = "rt_gpu_debug_light_pdf"


@pytest.fixture(scope="module")
def hc():
    return hs.hostcheck()


def host_pdfs(hc, sc, rays):
    m = len(rays)
    pe, pq = np.zeros(m, np.float32), np.zeros(m, np.float32)
    d = sc.desc()
    rc = hc.hc_light_pdf(C.byref(d), C.c_uint64(m), hs._ptr(rays), hs._ptr(pe), hs._ptr(pq))
    assert rc == 0, rc
    return pe, pq


def check(name, b, pdfs, floor):
    """Every path's pdfs within the bounds, and the scenario not vacuous."""
    msgs = []
    for label, pdf in pdfs.items():
        bad = b.wrong(pdf)
        print(f"{name} [{label}]: {len(pdf)} rays, tight {b.tight.mean():.3f}, clear {(b.n_clear > 0).mean():.3f}, "
              f"max clear hits {b.n_clear.max()}, out of bounds {int(bad.sum())}")
        if bad.any():
            msgs.append(b.report(f"{name} [{label}]", pdf))
    assert not msgs, "\n".join(msgs)
    assert b.tight.mean() >= floor, (name, b.tight.mean())


@pytest.mark.parametrize("name", sorted(ls.SCENARIOS))
def test_host_light_pdf_within_the_brute_force_bounds(name, hc):
    sc, rays = ls.make(name)
    b = ls.Bounds(hc, sc, rays)
    check(name, b, dict(zip(("exact", "q8"), host_pdfs(hc, sc, rays))), ls.TIGHT_FLOOR[name])
    if name in ls.BOX_SCENARIOS:
        miss, inside = ls.box_categories(sc, rays)
        empty = (b.n_clear == 0) & (b.n_border == 0)
        counts = int(miss.sum()), int((inside & empty).sum()), int((b.n_clear > 0).sum())
        print(f"{name}: rays missing the light box {counts[0]}, inside it without a light {counts[1]}, with clear hits {counts[2]}")
        assert min(counts) > 0, counts


@pytest.mark.parametrize("name", ls.GLTF_SCENES)
def test_host_light_pdf_on_the_gltf_rooms(name, hc, scene_dir):
    sc = gltf.load_gltf(scene_dir(name), 1.0)
    rays = ls.gltf_rays(sc, ls.GLTF_RAYS)
    b = ls.Bounds(hc, sc, rays)
    check(name, b, dict(zip(("exact", "q8"), host_pdfs(hc, sc, rays))), ls.TIGHT_FLOOR[name])


def test_scenarios_hit_their_edges(hc):
    """The scenarios build what their names say: dozens of lights along one ray, both copies of a duplicate, zero-area
    lights counted in n_lights, and the light chain's stack need (printed; the upload refuses it above
    RT_EXT_STACK_CAP)."""
    sc, rays = ls.make("layers")
    assert ls.Bounds(hc, sc, rays).n_clear.max() >= 30
    sc, rays = ls.make("duplicates")
    b = ls.Bounds(hc, sc, rays)
    assert (b.n_clear[b.tight] >= 2).any()
    sc, _ = ls.make("zero_area")
    lt = ls.light_tris(sc).astype(np.float64)
    zero = np.linalg.norm(np.cross(lt[:, 1] - lt[:, 0], lt[:, 2] - lt[:, 0]), axis=1) == 0
    assert zero.sum() == 500 and len(sc.light_bvh.objects) == 2500
    sc, _ = ls.make("chain")
    out = np.zeros(3)
    hc.hc_set_rebuild(1)
    try:
        rc = hc.hc_stack_need(C.byref(sc.desc()), hs._ptr(out))
    finally:
        hc.hc_set_rebuild(0)
    print(f"chain as lights: light BVH stack need {out[1]:.0f} (cap {out[2]:.0f}), pack_scene {rc}")
    assert rc in (0, next(code for code, n in _abi.STATUS.items() if n == "RT_ERR_BAD_SCENE"))
    assert (rc == 0) == (out[1] <= out[2])


def test_lights_off_the_ray_give_exactly_zero(hc):
    """Rays that start on a light and meet no other: their own light at t ~ 0 does not count."""
    sc, rays = ls.make("on_lights")
    b = ls.Bounds(hc, sc, rays)
    empty = (b.n_clear == 0) & (b.n_border == 0)
    assert empty.mean() > 0.2
    for pdf in host_pdfs(hc, sc, rays):
        assert (pdf[empty] == 0.0).all()


@pytest.mark.parametrize("name", sorted(ls.SCENARIOS))
def test_brute_force_matches_its_numpy_statement(name, hc):
    """hc_brute_light_pdf against the same rule written in numpy, on 300 rays of each scenario."""
    sc, rays = ls.make(name)
    rays = np.ascontiguousarray(rays[np.random.default_rng(2).choice(len(rays), 300, replace=False)])
    b = ls.Bounds(hc, sc, rays)
    lo, hi, nc, nb = ls.bounds_numpy(b.lights, rays, b.eps)
    assert np.array_equal(b.n_clear, nc) and np.array_equal(b.n_border, nb)
    assert np.allclose(b.lo, lo, rtol=1e-12, atol=0)
    # a borderline pair's cosine can be 1e-12 (grazing): the two statements form it in another order, and its term
    # carries that cancellation into hi
    fin = np.isfinite(hi)
    assert np.array_equal(np.isfinite(b.hi), fin) and np.allclose(b.hi[fin], hi[fin], rtol=1e-8, atol=0)


def test_brute_force_by_hand(hc):
    """A ray straight through two stacked unit lights 1 and 2 away (terms t^2 / A = 1 / 2 and 4 / 2; n_lights = 3 with
    a zero-area light), a ray through their shared edge with a third light (borderline), and a ray that misses."""
    sc = ls.light_scene(np.array([[[-1, -1, 0], [1, -1, 0], [-1, 1, 0]], [[-1, -1, -1], [1, -1, -1], [-1, 1, -1]],
                                  [[0, 0, 5], [0, 0, 5], [1, 0, 5]]], np.float32), [True, True, True])
    rays = np.array([[-0.5, -0.5, 1, 0, 0, -1], [0, 0, 1, 0, 0, -1], [5, 5, 1, 0, 0, -1]], np.float32)
    b = ls.Bounds(hc, sc, rays)
    assert b.n_clear.tolist() == [2, 0, 0] and b.n_border.tolist() == [0, 2, 0]
    assert b.lo[0] <= (0.5 + 2.0) / 3 <= b.hi[0] and b.hi[0] / b.lo[0] < 1 + 1e-4
    assert b.lo[1] == 0.0 and b.hi[1] > 0 and b.lo[2] == b.hi[2] == 0.0
    pe, pq = host_pdfs(hc, sc, rays)
    assert not b.wrong(pe).any() and not b.wrong(pq).any()


# ---- rt_gpu_debug_light_pdf without a device ------------------------------------------------------------------------------
def test_debug_entry_is_exported_and_declared():
    assert NAME in gpu.SYMBOLS
    getattr(C.CDLL(gpu.LIB_PATH), NAME)
    with open(os.path.join(ROOT, "include", "rt_gpu.h")) as f:
        assert f"int {NAME}(rt_gpu_ctx *ctx, uint64_t n, const float *rays, float *pdf);" in f.read()


def test_debug_entry_refuses_null_arguments():
    L = gpu.lib()
    bad = next(code for code, name in _abi.STATUS.items() if name == "RT_ERR_INVALID_ARG")
    rays, pdf = np.zeros((1, 6), np.float32), np.zeros(1, np.float32)
    assert L.rt_gpu_debug_light_pdf(None, 1, hs._ptr(rays), hs._ptr(pdf)) == bad
    assert L.rt_gpu_debug_light_pdf(None, 0, None, None) == bad
    assert NAME in L.rt_gpu_last_error().decode()


def test_no_device_refuses_the_handle():
    """Without a CUDA device there is no handle to ask (RT_ERR_NO_DEVICE), so RtGpu.debug_light_pdf cannot run."""
    if gpu.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_DEVICE"):
        gpu.RtGpu(1, 0)
