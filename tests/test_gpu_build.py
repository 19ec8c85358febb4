"""The device-side scene build (csrc/gpu_build.cuh; SURVEY.md 8(f)-2: BVH build on the GPU replacing BVH::build,
src/bvh.h:262-393).  The tree the library builds on the B200 is downloaded through the diagnostic entry
rt_gpu_debug_get_bvh and checked on the host: structural invariants, exact boxes, SAH cost against the host builder
(csrc/sah_build.h, the same algorithm), containment of the quantised 4-wide nodes, and — what parity is about — the
same primary ids and images as the host-built tree."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, golden_array
from hit_scenarios import check_tree, triangles_scene

import rt_b200
from rt_b200 import _abi, gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hc():
    return C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libhostcheck.so"))


def _download(rt):
    info = rt.debug_bvh(0, np.uint32)
    return info, rt.debug_bvh(1, _abi.NODE_DTYPE), rt.debug_bvh(2, np.uint32), rt.debug_bvh(3, np.uint8), rt.debug_bvh(4, np.uint8)


@pytest.mark.parametrize("name", ["tiny", "texall", "small_lights"])
def test_device_built_tree_small_scenes(name, rt, hc, manifest, golden_scene):
    sc = golden_scene(name)
    rt.upload_scene(sc)
    cost, depth, inner = check_tree(hc, sc, *_download(rt))
    m = manifest["scenes"][name]
    ids = rt.primary_ids(m["width"], m["height"])
    ref = golden_array(f"{name}_ids.i32", np.int32, (m["height"], m["width"]))
    assert (ids == ref).mean() >= 0.999


def test_device_built_tree_260k_scene(rt, hc, manifest, big_scene):
    """Same algorithm as csrc/sah_build.h: the SAH cost of the device tree is that of the host tree (the partition order
    inside a node differs, so the trees are not identical), and the images do not depend on the tree."""
    rt.upload_scene(big_scene)
    info, nodes, objects, qn, tris = _download(rt)
    cost, depth, inner = check_tree(hc, big_scene, info, nodes, objects, qn, tris)
    d = big_scene.desc()
    host = np.zeros(8)
    assert hc.hc_sah_stats(C.byref(d), host.ctypes.data_as(C.c_void_p)) == 0
    print(f"device tree: SAH cost {cost:.3f}, depth {depth:.0f}, {inner:.0f} inner, {info[2]} wide nodes, stack need {info[4]}, "
          f"{info[7]} top-down levels; host tree: cost {host[6]:.3f}, depth {host[4]:.0f}, {host[1]:.0f} inner")
    assert abs(cost - host[6]) / host[6] < 0.01
    m = manifest["scenes"]["big_lights"]
    w, h = m["ids_width"], m["ids_height"]
    ids = rt.primary_ids(w, h)
    ref = golden_array("big_lights_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999
    rt.render(200, 200, 8, seed=5)
    img_dev, st_dev = rt.readback()
    os.environ["RT_HOST_BUILD"] = "1"  # A/B: the same upload through the host builder
    try:
        rt.upload_scene(big_scene)
        assert rt.debug_bvh(0, np.uint32)[6] == 0
        ids_host = rt.primary_ids(w, h)
        rt.render(200, 200, 8, seed=5)
        img_host, st_host = rt.readback()
    finally:
        del os.environ["RT_HOST_BUILD"]
    assert (ids == ids_host).mean() >= 0.9999
    rel = np.abs(img_dev - img_host) / (np.abs(img_host) + 1e-3)
    assert (rel.max(axis=2) > 1e-3).mean() <= 0.01
    assert abs(st_dev["extension_rays"] - st_host["extension_rays"]) <= 1e-3 * st_host["extension_rays"]


def test_device_build_is_deterministic(rt, big_scene):
    rt.upload_scene(big_scene)
    a = _download(rt)
    rt.upload_scene(big_scene)
    b = _download(rt)
    n_slots = a[0][1]
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])  # info, triangle order
    assert a[3].tobytes() == b[3].tobytes() and a[4].tobytes() == b[4].tobytes()  # wide nodes, device triangles
    # binary nodes: compare the slots the tree uses (unused slots of the sparse layout are undefined)
    used = np.zeros(n_slots, bool)
    todo = [0]
    while todo:
        i = todo.pop()
        used[i] = True
        if a[1][i]["left_child"] != _abi.RT_NO_CHILD:
            todo += [int(a[1][i]["left_child"]), int(a[1][i]["right_child"])]
    assert a[1][used].tobytes() == b[1][used].tobytes()


@pytest.mark.parametrize("n", [1, 2, 9, 33, 1000])
def test_device_build_edge_cases(n, rt, hc):
    """One triangle, a handful, and n copies of the SAME triangle (all centroids coincide: binning cannot separate them,
    the builder splits by position until the leaves hold <= 8)."""
    one = [[-1, -1, 0], [1, -1, 0], [0, 1, 0]]
    sc = triangles_scene([one] * n)
    rt.upload_scene(sc)
    info, nodes, objects, qn, tris = _download(rt)
    assert info[0] == n and sorted(objects.tolist()) == list(range(n))
    d = sc.desc()
    out = np.zeros(8)
    assert hc.hc_tree_stats(C.byref(d), nodes.ctypes.data_as(C.c_void_p), C.c_uint64(len(nodes)), objects.ctypes.data_as(C.c_void_p),
                            C.c_uint64(len(objects)), out.ctypes.data_as(C.c_void_p)) == 0
    assert out[5] == 1.0 and out[3] <= 8
    ids = rt.primary_ids(32, 32)
    assert ids[16, 16] >= 0 and ids[0, 0] == -1
    # distinct triangles in a row: every one is found
    s = min(1.0, 4.0 / max(n - 1, 1))  # side scaled so that neighbours do not overlap: each centroid has one answer
    row = [[[x - 0.4 * s, -0.4 * s, 0], [x + 0.4 * s, -0.4 * s, 0], [x, 0.4 * s, 0]] for x in np.linspace(-2, 2, n)] if n > 1 else [one]
    sc = triangles_scene(row)
    rt.upload_scene(sc)
    info = rt.debug_bvh(0, np.uint32)
    assert info[0] == n and info[4] <= 96
    # one 1x1 view straight down onto each centroid (the pixel centre's camera term is 0: the ray is the camera's axis)
    centroids = np.asarray(row, np.float32).astype(np.float64).mean(axis=1)
    cams = [rt_b200.Camera((c[0], c[1], 5), (1, 0, 0), (0, 1, 0), (0, 0, -1), 1.0) for c in centroids]
    assert rt.primary_ids(1, 1, cameras=cams).reshape(-1).tolist() == list(range(n))


def test_device_build_rejects_non_finite_geometry(rt):
    tri = np.array([[[-1, -1, 0], [1, -1, 0], [0, 1, 0]]] * 40, np.float32)
    tri[7, 1, 0] = np.inf
    sc = triangles_scene(tri)
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_BAD_SCENE"):
        rt.upload_scene(sc)
    rt.upload_scene(triangles_scene(tri[:7]))  # the handle stays usable


def test_empty_scene_through_the_device_build(rt):
    sc = triangles_scene(np.zeros((0, 3, 3), np.float32))
    rt.upload_scene(sc)
    ids = rt.primary_ids(8, 8)
    assert (ids == -1).all()
    rt.render(8, 8, 4, seed=1)
    img, _ = rt.readback()
    assert np.allclose(img, np.asarray(sc.bg_color, np.float32)[None, None, :])
