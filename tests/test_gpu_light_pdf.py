"""Light pdfs of the kernels against the float64 brute force (hc_brute_light_pdf) on the scenarios of light_scenarios.py.
rt_gpu_debug_light_pdf hands the rays to the device as pending rays: in the default library through k_shade's own append
(the box of all lights: 0 on a miss, listed otherwise) and k_lightpdf_list, in librt_gpu_wide8.so through k_extend8's
light mode (a child pytest, as in test_eight_wide_build_keeps_parity).  Also the light side of rt_gpu_update_geometry
(light box, DLight records and light BVH of moved lights), the entry's refusals, and a scene without emitters."""
import os
import subprocess
import sys

import numpy as np
import pytest

import hit_scenarios as hs
import light_scenarios as ls
from test_gpu_update import lights_translated, moved
from test_light_pdf_host import check

from conftest import ROOT
from rt_b200 import _abi, gltf, gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hc():
    return hs.hostcheck()


def _lib():
    return os.path.basename(os.environ.get("RT_GPU_LIB", "librt_gpu.so"))


def _status(name):
    return next(code for code, n in _abi.STATUS.items() if n == name)


@pytest.mark.parametrize("name", sorted(ls.SCENARIOS))
def test_kernel_light_pdf_within_the_brute_force_bounds(name, rt, hc):
    sc, rays = ls.make(name)
    try:
        rt.upload_scene(sc)
    except gpu.RtGpuError as e:  # the light chain: a light BVH whose traversal needs more than RT_EXT_STACK_CAP entries
        assert name == "chain" and "RT_ERR_BAD_SCENE" in str(e), e
        print(f"{name} [{_lib()}]: upload refused: {e}")
        return
    b = ls.Bounds(hc, sc, rays)
    check(name, b, {_lib(): rt.debug_light_pdf(rays)}, ls.TIGHT_FLOOR[name])
    if name in ls.BOX_SCENARIOS:
        miss, inside = ls.box_categories(sc, rays)
        empty = (b.n_clear == 0) & (b.n_border == 0)
        counts = int(miss.sum()), int((inside & empty).sum()), int((b.n_clear > 0).sum())
        print(f"{name}: rays missing the light box {counts[0]}, inside it without a light {counts[1]}, with clear hits {counts[2]}")
        assert min(counts) > 0, counts


@pytest.mark.parametrize("name", ls.GLTF_SCENES)
def test_kernel_light_pdf_on_the_gltf_rooms(name, rt, hc, scene_dir):
    sc = gltf.load_gltf(scene_dir(name), 1.0)
    rays = ls.gltf_rays(sc, ls.GLTF_RAYS)
    rt.upload_scene(sc)
    check(name, ls.Bounds(hc, sc, rays), {_lib(): rt.debug_light_pdf(rays)}, ls.TIGHT_FLOOR[name])


def test_light_pdf_follows_geometry_updates(rt, hc, golden_scene):
    """small_lights with its lights translated, then teleported by 3e4: the light box, the DLight records and the light
    BVH after rt_gpu_update_geometry bound as the brute force of the moved lights says; updated back, the pdfs are the
    fresh upload's bit for bit.  (The 8-wide library refuses geometry updates by design.)"""
    A = golden_scene("small_lights").without_scene_bvh()
    rng = np.random.default_rng(11)
    rt.upload_scene(A)
    em = (A.materials["emission"][A.tri_material] != 0).any(axis=1)
    translated = lights_translated(A)
    far = translated.tri_pos.astype(np.float64)
    far[em] += [3e4, -3e4, 3e4]
    steps = [("translated", translated), ("teleported", moved(A, far))]
    fresh = None
    for label, B in [("upload", A)] + steps:
        if label != "upload":
            rt.update_geometry(B)
        lights = ls.light_tris(B)
        rays = np.concatenate([hs.targeted(rng, lights, 3000, 0.05, 2.0), hs.beside(rng, lights, 1000, 0.05, 2.0),
                               ls.from_surface(rng, lights, 1000), ls.signed_zero_axis(rng, lights.reshape(-1, 3)[rng.choice(3 * len(lights), 1000)])])
        rays = np.ascontiguousarray(rays, np.float32)
        b = ls.Bounds(hc, B, rays)
        pdf = rt.debug_light_pdf(rays)
        check(f"small_lights {label}", b, {_lib(): pdf}, 0.3)
        if label == "upload":
            fresh = (rays, pdf)
    rt.update_geometry(A)
    assert rt.debug_light_pdf(fresh[0]).tobytes() == fresh[1].tobytes()


def test_scene_without_emitters_gives_zeros(rt):
    sc = hs.triangles_scene(hs._soup(np.random.default_rng(3), 200, 1e-2, 0.3))
    rt.upload_scene(sc)
    rays = hs.random_rays(np.random.default_rng(4), -1, 1, 500)
    assert (rt.debug_light_pdf(rays) == 0).all() and len(rt.debug_light_pdf(rays[:0])) == 0


def test_refusals(golden_scene):
    rays, pdf = np.zeros((2, 6), np.float32), np.zeros(2, np.float32)
    with gpu.RtGpu(1, 0) as g:
        L = gpu.lib()
        call = lambda r, p: L.rt_gpu_debug_light_pdf(g._h, 2, hs._ptr(r) if r is not None else None, hs._ptr(p) if p is not None else None)
        assert call(rays, pdf) == _status("RT_ERR_NO_SCENE")
        g.upload_scene(golden_scene("small_lights"))
        assert call(None, pdf) == _status("RT_ERR_INVALID_ARG")
        assert call(rays, None) == _status("RT_ERR_INVALID_ARG")
        from rt_b200 import textscene

        g.upload_text_scene(textscene.TextScene())
        assert call(rays, pdf) == _status("RT_ERR_INVALID_ARG")


def test_eight_wide_build_light_pdf():
    """The same scenarios through librt_gpu_wide8.so (k_extend8's light mode over the 8-wide light BVH) in a fresh
    interpreter; the update case is left out (that library refuses geometry updates)."""
    if os.environ.get("RT_GPU_LIB"):
        pytest.skip("already running an alternative build")
    lib = os.path.join(ROOT, "raytracing-course-hw-public_b200", "librt_gpu_wide8.so")
    env = dict(os.environ, RT_GPU_LIB=lib)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", "-m", "gpu", os.path.abspath(__file__),
                        "-k", "not updates"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-8000:])
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
