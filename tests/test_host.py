"""Host-side logic, no GPU: C-ABI libraries load and export what include/*.h declares, the Python loader and
the own BVH build reproduce the reference's flattened scene bit for bit, RTSC round trips, the re-packed
device layout traverses to the same ids, and the device math header (compiled for the host, test-only)
follows the oracle path by path."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import oracle_lib as O
from conftest import GOLDEN, ROOT, golden_array
from scene_digest import SECTIONS, flattening_digest

import rt_b200
from rt_b200 import _abi, gltf, gpu, host

SMALL = ["tiny", "texall", "small_lights"]


def assert_same_scene(a, b):
    for x, y, name in zip(a._sections(), b._sections(), SECTIONS):
        assert (x is None) == (y is None), name
        if x is not None:
            assert x.tobytes() == y.tobytes(), name
    for k in ("camera_position", "camera_right", "camera_up", "camera_forward", "fov_x", "bg_color", "eps",
              "min_roughness", "vndf_factor"):
        assert np.array_equal(np.asarray(getattr(a, k)), np.asarray(getattr(b, k))), k
    assert a.ray_depth == b.ray_depth and a.env_texture == b.env_texture
    assert a.scene_bvh.root == b.scene_bvh.root and a.light_bvh.root == b.light_bvh.root


def declared_symbols(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rt_(?:gpu|host|scene|text_scene)_\w+)\s*\(", text)))


def test_c_abi_exports_every_declared_symbol():
    for header, mod in (("rt_gpu.h", gpu), ("rt_host.h", host)):
        declared = declared_symbols(header)
        assert declared, header
        assert sorted(mod.SYMBOLS) == declared, (header, declared)
        L = C.CDLL(mod.LIB_PATH)
        for s in declared:
            assert hasattr(L, s), s
    assert gpu.lib().rt_gpu_abi_version() == _abi.RT_GPU_ABI_VERSION


def test_struct_sizes_match_header():
    assert C.sizeof(_abi.rt_bvh_node) == 40
    assert C.sizeof(_abi.rt_bvh_desc) == 32
    assert C.sizeof(_abi.rt_camera) == 52
    assert C.sizeof(_abi.rt_render_params) == 48  # + pixel_begin, pixel_end (image-tile split)
    # rt_scene_desc: 8 + 52 + 12 + 12 + 4 + 12 (+pad) ... checked through a C round trip instead
    sc = rt_b200.SceneData.load(os.path.join(GOLDEN, "tiny.rtsc"))
    assert host.validate(sc) == 0


def test_no_cpu_fallback_without_a_device():
    """The product fails loudly when no CUDA device is usable (in a child process that sees none, so that this runs on
    a machine with a GPU as well)."""
    import subprocess
    import sys

    code = ("import sys; sys.path.insert(0, sys.argv[1]); import rt_b200; from rt_b200 import gpu\n"
            "try:\n    gpu.RtGpu(1, 0)\nexcept gpu.RtGpuError as e:\n    print(e)\n    sys.exit(0)\nsys.exit(1)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "RT_ERR_NO_DEVICE" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("name", SMALL)
def test_python_loader_and_bvh_build_match_reference_flattening(name, scene_dir, manifest, golden_scene):
    m = manifest["scenes"][name]
    mine = gltf.load_gltf(scene_dir(name), m["width"] / m["height"])
    assert_same_scene(golden_scene(name), mine)


def test_texmaps_loader_matches_reference_flattening(scene_dir, manifest, golden_scene):
    m = manifest["scenes"]["texmaps"]
    assert_same_scene(golden_scene("texmaps"), gltf.load_gltf(scene_dir("texmaps"), m["width"] / m["height"]))


@pytest.mark.parametrize("name", ["tiny_lt", "small_lights_lt"])
def test_extra_light_triangle_matches_reference_flattening(name, scene_dir, manifest, golden_scene):
    """ADD_LIGHT_TRIANGLE (config.h:39-47, false at HEAD): the object parse_gltf_scene appends under that switch
    (scene.h:479-498) — the Python loader's run-time form of it reproduces the reference's flattened scene bit for bit
    (positions, its own normal, default material with emission 10, both BVHs with the triangle in them)."""
    m = manifest["scenes"][name]
    ref = golden_scene(name)
    base = golden_scene(m["base"])
    mine = gltf.load_gltf(scene_dir(m["base"]), m["width"] / m["height"], add_light_triangle=True)
    assert_same_scene(ref, mine)
    assert ref.n_tris == base.n_tris + 1 and len(ref.light_bvh.objects) == len(base.light_bvh.objects) + 1
    lt = ref.tri_pos[-1]
    cam_z = (lt - ref.camera_position) @ ref.camera_forward
    assert np.allclose(cam_z, -0.1, atol=1e-5)  # 0.1 behind the camera plane
    assert np.all(ref.materials[ref.tri_material[-1]]["emission"] == 10.0)
    os.environ["RT_ADD_LIGHT_TRIANGLE"] = "1"  # the environment switch of the CLIs
    try:
        assert_same_scene(ref, gltf.load_gltf(scene_dir(m["base"]), m["width"] / m["height"]))
    finally:
        del os.environ["RT_ADD_LIGHT_TRIANGLE"]


def test_environment_map_loader_matches_reference_flattening(scene_dir, manifest, golden_scene):
    """Scene::bg as an equirectangular texture (main.cpp:29-31): the Python loader appends it exactly like the
    reference-hosted flattener; the RTSC container carries env_texture."""
    m = manifest["scenes"]["tiny_env"]
    mine = gltf.load_gltf(scene_dir("tiny"), m["width"] / m["height"], env_map=os.path.join(GOLDEN, m["env_map"]))
    ref = golden_scene("tiny_env")
    assert ref.env_texture == 1 and mine.env_texture == ref.env_texture
    assert_same_scene(ref, mine)
    white = gltf.load_gltf(scene_dir("tiny"), 1.0)
    assert white.env_texture == 0 and len(white.textures) == len(mine.textures) - 1
    d = ref.desc()
    d.env_texture = 7
    assert host.lib().rt_scene_validate(C.byref(d)) == -7  # RT_ERR_BAD_SCENE: env_texture > n_textures


def test_big_scene_flattening_matches_reference(scene_dir, big_scene, tmp_path):
    """The reference's flattening of the 260 192-triangle scene, pinned by digests of its dump; compared with the dump
    itself as well where oracle/_ref was built."""
    with open(os.path.join(GOLDEN, "big_lights_flat.json")) as f:
        ref = json.load(f)
    assert flattening_digest(big_scene) == {k: ref[k] for k in ("n_tris", "sections", "fields")}
    assert big_scene.n_tris == 260192
    if O.have_ref_tool():
        out = tmp_path / "big.rtsc"
        O.ref_tool("dump", scene_dir("big_lights"), 64, 64, out)
        assert_same_scene(rt_b200.SceneData.load(str(out)), big_scene)


def test_bvh_build_edge_cases():
    empty = host.build_bvh(np.zeros((0, 9), np.float32))
    assert empty.root == _abi.RT_NO_CHILD and len(empty.nodes) == 0
    one = host.build_bvh(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32))
    assert len(one.nodes) == 1 and one.nodes[0]["obj_end"] == 1 and one.root == 0
    tri = np.tile(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32), (50, 1))  # identical centroids: one big leaf
    same = host.build_bvh(tri)
    assert len(same.nodes) == 1 and same.nodes[0]["obj_end"] == 50
    none_selected = host.build_bvh(tri, select=np.zeros(50, np.uint8))
    assert none_selected.root == _abi.RT_NO_CHILD


def test_rtsc_round_trip(tmp_path, golden_scene):
    sc = golden_scene("texall")
    p = tmp_path / "a.rtsc"
    sc.save(str(p))
    assert_same_scene(sc, rt_b200.SceneData.load(str(p)))
    # C writer/reader agree with the Python ones
    d = sc.desc()
    q = tmp_path / "b.rtsc"
    assert host.lib().rt_scene_save(C.byref(d), os.fsencode(str(q))) == 0
    assert open(p, "rb").read() == open(q, "rb").read()
    out = C.POINTER(_abi.rt_scene_desc)()
    L = host.lib()
    L.rt_scene_load.argtypes = [C.c_char_p, C.POINTER(C.POINTER(_abi.rt_scene_desc))]
    L.rt_scene_free.argtypes = [C.POINTER(_abi.rt_scene_desc)]
    assert L.rt_scene_load(os.fsencode(str(q)), C.byref(out)) == 0
    assert out.contents.n_tris == sc.n_tris and out.contents.scene_bvh.n_nodes == len(sc.scene_bvh.nodes)
    L.rt_scene_free(out)


def test_bad_scene_is_rejected(golden_scene):
    sc = rt_b200.SceneData.load(os.path.join(GOLDEN, "tiny.rtsc"))
    sc.tri_material = sc.tri_material.copy()
    sc.tri_material[0] = 99
    assert host.validate(sc) == -7  # RT_ERR_BAD_SCENE


def test_host_tonemap_matches_reference():
    x = golden_array("tonemap_in.f32", np.float32)
    assert np.array_equal(host.tonemap_rgb8(x.reshape(-1, 3)).reshape(-1), golden_array("tonemap_out.u8", np.uint8))


# ---- device math compiled for the host (tests/hostcheck, test-only) --------------------------------------
@pytest.fixture(scope="module")
def hc():
    L = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libhostcheck.so"))
    return L


@pytest.mark.parametrize("name", SMALL)
def test_repacked_traversal_gives_reference_ids(name, hc, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    ids = np.zeros((h, w), np.int32)
    assert hc.hc_primary_ids(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p)) == 0
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999


@pytest.mark.parametrize("name", SMALL)
def test_quantised_node_traversal_gives_reference_ids(name, hc, manifest, golden_scene):
    """k_extend's per-ray arithmetic (32-byte quantised nodes, fused o/d slab test) finds the reference's hits."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    ids = np.zeros((h, w), np.int32)
    assert hc.hc_primary_ids_q(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p)) == 0
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999


def _qnode_check(hc, scene):
    d = scene.desc()
    out = (C.c_double * 5)()
    assert hc.hc_qnode_check(C.byref(d), out) == 0
    return list(out)


@pytest.mark.parametrize("name", SMALL)
def test_quantised_nodes_are_conservative(name, hc, golden_scene):
    n, bad, tight, area_exact, area_q = _qnode_check(hc, golden_scene(name))
    assert n > 0 and bad == 0 and tight == 0
    assert area_q >= area_exact


def test_quantised_nodes_are_conservative_on_the_260k_scene(hc, big_scene):
    n, bad, tight, area_exact, area_q = _qnode_check(hc, big_scene)
    assert n > 70000 and bad == 0 and tight == 0
    # 8 bits per plane on a per-node grid: the decoded boxes are only a few percent larger
    assert 1.0 <= area_q / area_exact < 1.10
    ids_q = np.zeros((96, 96), np.int32)
    ids = np.zeros((96, 96), np.int32)
    d = big_scene.desc()
    assert hc.hc_primary_ids_q(C.byref(d), 96, 96, ids_q.ctypes.data_as(C.c_void_p)) == 0
    assert hc.hc_primary_ids(C.byref(d), 96, 96, ids.ctypes.data_as(C.c_void_p)) == 0
    assert (ids_q == ids).mean() >= 0.999


# ---- the library's own SAH builder (csrc/sah_build.h) ------------------------------------------------------
@pytest.mark.parametrize("name", SMALL)
def test_sah_rebuilt_tree_gives_reference_ids(name, hc, manifest, golden_scene):
    """Closest hits do not depend on the tree: traversal of the library-built BVH (both node formats) finds the
    reference's primary ids."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    hc.hc_set_rebuild(1)
    try:
        for fn in (hc.hc_primary_ids, hc.hc_primary_ids_q):
            ids = np.zeros((h, w), np.int32)
            assert fn(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p)) == 0
            assert (ids == ref).mean() >= 0.999
        out = (C.c_double * 5)()
        assert hc.hc_qnode_check(C.byref(d), out) == 0 and out[1] == 0 and out[2] == 0
    finally:
        hc.hc_set_rebuild(0)


def test_sah_builder_invariants_on_the_260k_scene(hc, big_scene):
    d = big_scene.desc()
    out = (C.c_double * 8)()
    assert hc.hc_sah_stats(C.byref(d), out) == 0
    secs, inner, leaves, max_leaf, max_depth, ok, cost, layout = list(out)
    print(f"sah build: {secs * 1e3:.0f} ms, {inner:.0f} inner, {leaves:.0f} leaves, max leaf {max_leaf:.0f}, depth {max_depth:.0f}, SAH cost {cost:.2f}")
    assert ok == 1.0 and layout == 1.0  # every triangle exactly once, every box the exact union of what is below it
    assert inner == leaves - 1 and max_leaf <= 8 and max_depth < 62
    hc.hc_set_rebuild(1)
    try:
        ids = np.zeros((96, 96), np.int32)
        ids_q = np.zeros((96, 96), np.int32)
        assert hc.hc_primary_ids(C.byref(d), 96, 96, ids.ctypes.data_as(C.c_void_p)) == 0
        assert hc.hc_primary_ids_q(C.byref(d), 96, 96, ids_q.ctypes.data_as(C.c_void_p)) == 0
    finally:
        hc.hc_set_rebuild(0)
    host_tree = np.zeros((96, 96), np.int32)
    assert hc.hc_primary_ids(C.byref(d), 96, 96, host_tree.ctypes.data_as(C.c_void_p)) == 0
    assert (ids == host_tree).mean() >= 0.999 and (ids_q == host_tree).mean() >= 0.999


@pytest.mark.parametrize("rebuild", [0, 1])
@pytest.mark.parametrize("name", SMALL)
def test_four_wide_collapse_gives_reference_ids(name, rebuild, hc, manifest, golden_scene):
    """k_extend's 4-wide mode (QNode4 = two binary levels per step, children sorted by entry distance)."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    ids = np.zeros((h, w), np.int32)
    steps = (C.c_uint64 * 2)()
    hc.hc_set_rebuild(rebuild)
    try:
        assert hc.hc_primary_ids_q4(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p), steps) == 0
    finally:
        hc.hc_set_rebuild(0)
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999
    assert steps[0] <= steps[1]  # never more node steps than the binary traversal


def test_rays_inside_the_plane_of_a_flat_node_keep_their_hits(hc, big_scene):
    """Light-sampled directions from one emissive panel to the next run INSIDE the panels' common plane (|d.y| ~ 1e-7,
    origin one ulp above it): the ray-space offset of the quantised slab test then carries an error of several units of
    t (it did with fma(org, 1/d, -o/d); (org - o)/d shrinks it), and a flat node's box has to absorb it.  The power-of-two grid does (its origin is
    rounded down to 14 mantissa bits, which leaves every flat box ~2e-6 of slack); an exact-cell variant tried in round 2
    lost 33 of 15 176 path-traced rays exactly here (DESIGN.md, k_extend).  Every hit the exact boxes find must be
    found through the quantised 4-wide nodes as well."""
    sc = big_scene
    lights = np.asarray(sc.light_bvh.objects, np.int64)
    assert len(lights) >= 8
    rng = np.random.default_rng(5)
    tri = sc.tri_pos[lights].astype(np.float64)  # (n, 3, 3)

    def points(idx):
        u, v = rng.random(len(idx)), rng.random(len(idx))
        flip = u + v > 1
        u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
        t = tri[idx]
        return t[:, 0] + (t[:, 1] - t[:, 0]) * u[:, None] + (t[:, 2] - t[:, 0]) * v[:, None]

    n = 4000
    a, b = rng.integers(0, len(lights), n), rng.integers(0, len(lights), n)
    o, q = points(a), points(b)
    keep = np.linalg.norm(q - o, axis=1) > 0.5
    o, q = o[keep], q[keep]
    o32 = o.astype(np.float32)
    o32[:, 1] = np.nextafter(o32[:, 1], np.float32(np.inf))  # one ulp above the panels' plane, like a hit point
    d = q - o32.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.ascontiguousarray(np.concatenate([o32, d.astype(np.float32)], axis=1), np.float32)
    m = len(rays)
    te, tq = np.zeros(m, np.float32), np.zeros(m, np.float32)
    ie, iq = np.zeros(m, np.int32), np.zeros(m, np.int32)
    desc = sc.desc()
    hc.hc_set_rebuild(1)
    try:
        assert hc.hc_trace_rays(C.byref(desc), C.c_uint64(m), rays.ctypes.data_as(C.c_void_p), ie.ctypes.data_as(C.c_void_p),
                                te.ctypes.data_as(C.c_void_p), iq.ctypes.data_as(C.c_void_p), tq.ctypes.data_as(C.c_void_p)) == 0
    finally:
        hc.hc_set_rebuild(0)
    assert (ie >= 0).mean() > 0.5  # these rays do hit something (walls, columns, other panels)
    lost = (ie >= 0) & ((iq < 0) | (tq > te * (1 + 1e-4)))
    assert lost.sum() == 0, f"{int(lost.sum())} of {m} in-plane rays lose their hit through the quantised nodes"


def test_four_wide_collapse_on_the_260k_scene(hc, big_scene):
    d = big_scene.desc()
    ids4 = np.zeros((96, 96), np.int32)
    ids2 = np.zeros((96, 96), np.int32)
    steps = (C.c_uint64 * 2)()
    hc.hc_set_rebuild(1)
    try:
        assert hc.hc_primary_ids_q4(C.byref(d), 96, 96, ids4.ctypes.data_as(C.c_void_p), steps) == 0
        assert hc.hc_primary_ids_q(C.byref(d), 96, 96, ids2.ctypes.data_as(C.c_void_p)) == 0
    finally:
        hc.hc_set_rebuild(0)
    assert (ids4 == ids2).mean() >= 0.999
    assert steps[0] < 0.6 * steps[1]  # measured 0.53: the collapse nearly halves the node steps


@pytest.mark.parametrize("rebuild", [0, 1])
@pytest.mark.parametrize("name", SMALL)
def test_eight_wide_traversal_gives_reference_ids(name, rebuild, hc, manifest, golden_scene):
    """The 8-wide collapse (QNode8: octant-ordered slots, group stack, re-ordered triangles) finds the reference's hits
    and holds every triangle exactly once."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    sc = golden_scene(name)
    d = sc.desc()
    ids = np.zeros((h, w), np.int32)
    out = (C.c_double * 4)()
    hc.hc_set_rebuild(rebuild)
    try:
        assert hc.hc_wide8_stats(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p), out) == 0
    finally:
        hc.hc_set_rebuild(0)
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999
    assert int(out[3]) == d.n_tris


@pytest.mark.parametrize("width,upload_path,rebuild", [(4, 0, 0), (4, 0, 1), (4, 1, 1), (8, 0, 0), (8, 0, 1)])
@pytest.mark.parametrize("name", SMALL + ["big"])
def test_wide_nodes_contain_their_triangles(name, width, upload_path, rebuild, hc, golden_scene, big_scene):
    """Containment invariant of QNode4 / QNode8, whatever built, collapsed and quantised the tree: every decoded child
    box holds every vertex of every triangle below it, and the tree reaches every triangle (scene + light BVH) once."""
    sc = big_scene if name == "big" else golden_scene(name)
    d = sc.desc()
    out = (C.c_double * 3)()
    hc.hc_set_rebuild(rebuild)
    try:
        assert hc.hc_wide_containment(C.byref(d), width, upload_path, out) == 0
    finally:
        hc.hc_set_rebuild(0)
    assert out[0] > 0
    assert out[1] == 0
    assert int(out[2]) == d.n_tris + d.light_bvh.n_objects


@pytest.mark.parametrize("name", SMALL)
def test_upload_path_packing_gives_reference_ids(name, hc, manifest, golden_scene):
    """rt_gpu_upload_scene's packing (library-built tree, direct parallel 4-wide collapse without the binary node array)
    finds the reference's hits."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    ids = np.zeros((h, w), np.int32)
    out = (C.c_double * 2)()
    assert hc.hc_primary_ids_upload_path(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p), out) == 0
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999


@pytest.mark.parametrize("name", SMALL)
def test_scene_without_host_bvh_is_built_by_the_library(name, hc, manifest, golden_scene):
    """rt_scene_desc.scene_bvh is optional (n_nodes == 0): the library builds the tree over all triangles in
    scene.objects order, so a host can skip BVH::build (bvh.h:262-393) for the scene."""
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).without_scene_bvh().desc()
    assert d.scene_bvh.n_nodes == 0 and d.scene_bvh.n_objects == 0
    ids = np.zeros((h, w), np.int32)
    out = (C.c_double * 2)()
    assert hc.hc_primary_ids_upload_path(C.byref(d), w, h, ids.ctypes.data_as(C.c_void_p), out) == 0
    ref = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    assert (ids == ref).mean() >= 0.999 and out[0] > 0
    res = np.zeros(8)
    assert hc.hc_wide_containment(C.byref(d), 4, 1, res.ctypes.data_as(C.c_void_p)) == 0
    assert res[0] > 0 and res[1] == 0 and res[2] >= golden_scene(name).n_tris  # planes checked, none violated, every triangle reached


def test_upload_path_packing_on_the_260k_scene(hc, big_scene):
    """Same wide tree as the serial collapse over the binary node array: same number of nodes, same node steps, same ids."""
    d = big_scene.desc()
    ids_a = np.zeros((96, 96), np.int32)
    ids_b = np.zeros((96, 96), np.int32)
    out = (C.c_double * 2)()
    steps = (C.c_uint64 * 2)()
    assert hc.hc_primary_ids_upload_path(C.byref(d), 96, 96, ids_a.ctypes.data_as(C.c_void_p), out) == 0
    hc.hc_set_rebuild(1)
    try:
        assert hc.hc_primary_ids_q4(C.byref(d), 96, 96, ids_b.ctypes.data_as(C.c_void_p), steps) == 0
    finally:
        hc.hc_set_rebuild(0)
    assert (ids_a == ids_b).all()
    assert abs(out[1] * 96 * 96 - steps[0]) < 0.5


def test_eight_wide_collapse_on_the_260k_scene(hc, big_scene):
    d = big_scene.desc()
    ids8 = np.zeros((96, 96), np.int32)
    ids2 = np.zeros((96, 96), np.int32)
    out = (C.c_double * 4)()
    steps = (C.c_uint64 * 2)()
    hc.hc_set_rebuild(1)
    try:
        assert hc.hc_wide8_stats(C.byref(d), 96, 96, ids8.ctypes.data_as(C.c_void_p), out) == 0
        assert hc.hc_primary_ids_q4(C.byref(d), 96, 96, ids2.ctypes.data_as(C.c_void_p), steps) == 0
    finally:
        hc.hc_set_rebuild(0)
    assert (ids8 == ids2).mean() >= 0.999
    assert int(out[3]) == d.n_tris
    assert out[1] > 4.0  # children per wide node (measured 4.5: the bottom of the tree holds quads, 2 triangles per leaf)
    assert out[2] * 96 * 96 < 0.8 * steps[0]  # fewer node steps than the 4-wide traversal of the same rays


def _comb_scene(levels, r=0.97):
    """Adversarial host tree (ADVICE r1): a comb N_k = (S_k, N_k+1) whose side branch S_k = (T, T') is larger than the
    rest of the chain, so the 4-wide collapse opens S_k and T and leaves N_k+1 one BINARY level below its wide
    parent: every wide node on the chain has four children (three pushes) and the wide depth equals the chain length."""
    tris, nodes = [], []

    def leaf(size, z):
        tris.append([[-size, -size, z], [size, -size, z], [0, size, z]])
        nodes.append(dict(lo=[-size, -size, z], hi=[size, size, z], l=_abi.RT_NO_CHILD, r=_abi.RT_NO_CHILD,
                          b=len(tris) - 1, e=len(tris)))
        return len(nodes) - 1

    def inner(make_l, make_r):
        i = len(nodes)
        nodes.append(None)
        l, rr = make_l(), make_r()
        lo = np.minimum(nodes[l]["lo"], nodes[rr]["lo"])
        hi = np.maximum(nodes[l]["hi"], nodes[rr]["hi"])
        nodes[i] = dict(lo=lo, hi=hi, l=l, r=rr, b=0, e=0)
        return i

    def chain(k):
        size, z = r ** k, 0.001 * k
        if k == levels:
            return leaf(size, z)
        pair = lambda dz: (lambda: inner(lambda: leaf(size, z + dz), lambda: leaf(size * 0.999, z + dz + 1e-4)))
        return inner(lambda: inner(pair(2e-4), pair(4e-4)), lambda: chain(k + 1))

    root = chain(0)
    arr = np.zeros(len(nodes), _abi.NODE_DTYPE)
    for i, nd in enumerate(nodes):
        arr[i] = (nd["lo"], nd["hi"], nd["l"], nd["r"], nd["b"], nd["e"])
    n = len(tris)
    sc = rt_b200.SceneData.load(os.path.join(GOLDEN, "tiny.rtsc"))
    sc.tri_pos = np.array(tris, np.float32)
    sc.tri_normals = np.tile(np.array([0, 0, 1], np.float32), (n, 3, 1))
    sc.tri_uv = np.zeros((n, 3, 2), np.float32)
    sc.tri_tangents = None
    sc.tri_material = np.zeros(n, np.uint32)
    sc.scene_bvh = _abi.BvhData(arr, np.arange(n, dtype=np.uint32), root)
    sc.light_bvh = _abi.BvhData(np.zeros(0, _abi.NODE_DTYPE), np.zeros(0, np.uint32), _abi.RT_NO_CHILD)
    return sc


def test_traversal_stack_bound_is_enforced_at_upload(hc, big_scene, golden_scene):
    """k_extend's per-ray stack holds RT_EXT_STACK_CAP entries without a bounds check; the packer computes the exact
    worst case of the collapsed tree and rejects what does not fit (a host tree may be 64 levels deep, bvh.h:371)."""
    out = np.zeros(3)
    hc.hc_set_rebuild(0)
    d = _comb_scene(30).desc()  # 30 chain levels x 3 pushes: fits
    assert hc.hc_stack_need(C.byref(d), out.ctypes.data_as(C.c_void_p)) == 0
    assert 85 <= out[0] <= out[2] == 96, out
    d = _comb_scene(58).desc()  # 61 binary levels (bvh.h:371 allows 64): three entries per level do not fit
    assert hc.hc_stack_need(C.byref(d), out.ctypes.data_as(C.c_void_p)) == -7  # RT_ERR_BAD_SCENE
    assert out[0] > 120, out
    hc.hc_set_rebuild(1)  # the library's own builder on the bench scene: far below the capacity
    d = big_scene.desc()
    assert hc.hc_stack_need(C.byref(d), out.ctypes.data_as(C.c_void_p)) == 0
    assert 0 < out[0] <= 64, out
    hc.hc_set_rebuild(0)
    d = golden_scene("small_lights").desc()
    assert hc.hc_stack_need(C.byref(d), out.ctypes.data_as(C.c_void_p)) == 0 and out[1] > 0


def test_device_philox_matches_known_answers(hc):
    out = (C.c_uint32 * 4)()
    hc.hc_philox((C.c_uint32 * 4)(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344),
                 (C.c_uint32 * 2)(0xA4093822, 0x299F31D0), out)
    assert list(out) == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


@pytest.mark.parametrize("name", SMALL)
def test_device_hit_data_matches_reference(name, hc, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"], m["height"]
    d = golden_scene(name).desc()
    info = np.zeros((h, w, 18), np.float32)
    assert hc.hc_hitinfo(C.byref(d), w, h, info.ctypes.data_as(C.c_void_p)) == 0
    ref = golden_array(f"{name}_hitinfo.f32", np.float32, (h, w, 18))
    ids = golden_array(f"{name}_ids.i32", np.int32, (h, w))
    hit = ids >= 0
    diff = np.abs(info - ref)[hit]
    diff[:, 16] = 0  # is_inside is folded into the normals
    diff[:, 0] /= np.maximum(ref[hit][:, 0], 1.0)  # t relative
    assert np.quantile(diff, 0.999) < 1e-4
    assert diff.max() < 5e-3


@pytest.mark.parametrize("name,tol_frac", [("tiny", 0.01), ("small_lights", 0.02)])
def test_device_math_follows_oracle_paths_eight_wide(name, tol_frac, hc, manifest, golden_scene):
    """The same path-by-path comparison with the scene packed in the 8-wide format (own triangle order, light pdf summed
    over the 8-wide light BVH)."""
    hc.hc_set_rebuild(1)
    hc.hc_set_wide8(1)
    try:
        _follow_oracle_paths(name, tol_frac, hc, manifest, golden_scene)
    finally:
        hc.hc_set_rebuild(0)
        hc.hc_set_wide8(0)


@pytest.mark.parametrize("rebuild", [0, 1])
@pytest.mark.parametrize("name,tol_frac", [("tiny", 0.01), ("small_lights", 0.02), ("tiny_env", 0.01), ("texmaps", 0.01),
                                           ("tiny_lt", 0.01), ("small_lights_lt", 0.04)])
def test_device_math_follows_oracle_paths(name, tol_frac, rebuild, hc, manifest, golden_scene):
    """Same Philox keys -> same paths: per-pixel means agree to float noise for all but the few pixels where a
    rounding difference flipped a discrete decision.  `rebuild`: with the library's own SAH tree instead of the
    host's (triangle attributes follow the packed order)."""
    hc.hc_set_rebuild(rebuild)
    try:
        _follow_oracle_paths(name, tol_frac, hc, manifest, golden_scene)
    finally:
        hc.hc_set_rebuild(0)


def _follow_oracle_paths(name, tol_frac, hc, manifest, golden_scene):
    m = manifest["scenes"][name]
    w, h = m["width"] // 2, m["height"] // 2
    sc = golden_scene(name)
    d = sc.desc()
    spp, seed = 16, 99
    out = np.zeros((h, w, 3), np.float32)
    cnt = (C.c_uint64 * 2)()
    assert hc.hc_render(C.byref(d), w, h, spp, 0, spp, C.c_uint64(seed), out.ctypes.data_as(C.c_void_p), cnt) == 0
    ref, st = O.render(sc, w, h, spp, rng_mode=O.RNG_PHILOX, seed=seed)
    rel = (np.abs(out - ref) / (np.abs(ref) + 1e-3)).max(axis=2)
    assert (rel > 1e-3).mean() <= tol_frac
    assert abs(np.mean(out) - np.mean(ref)) < 2e-3 * np.mean(ref)
    assert abs(cnt[0] - st["extension_rays"]) <= 0.02 * st["extension_rays"]


def test_many_lights_scene_follows_oracle_paths(hc, scene_dir):
    """1152 emissive triangles (a light BVH five wide levels deep, every bounce samples and queries it): the host
    compilation of the device math follows the pinned oracle path by path, like the GPU test of the same scene."""
    from rt_b200 import gltf

    sc = gltf.load_gltf(scene_dir("small_manylights"), 1.0)
    assert len(sc.light_bvh.objects) == 1152
    d = sc.desc()
    w, h, spp, seed = 48, 36, 8, 5
    out = np.zeros((h, w, 3), np.float32)
    cnt = (C.c_uint64 * 2)()
    assert hc.hc_render(C.byref(d), w, h, spp, 0, spp, C.c_uint64(seed), out.ctypes.data_as(C.c_void_p), cnt) == 0
    ref, st = O.render(sc, w, h, spp, rng_mode=O.RNG_PHILOX, seed=seed)
    rel = (np.abs(out - ref) / (np.abs(ref) + 1e-3)).max(axis=2)
    assert (rel > 1e-3).mean() <= 0.08
    assert abs(np.mean(out) - np.mean(ref)) < 5e-3 * np.mean(ref)
    assert abs(cnt[0] - st["extension_rays"]) <= 0.02 * st["extension_rays"]


# ---- CLI surface (src/main.cpp:16-49) ---------------------------------------------------------------------
CLI = os.path.join(ROOT, "bin", "raytracer_b200")


@pytest.mark.skipif(not os.path.exists(CLI), reason="reference-hosted CLI not built (reference sources absent)")
def test_cli_argument_errors_match_reference():
    import subprocess

    r = subprocess.run([CLI, "a", "b"], capture_output=True, text=True)
    assert r.returncode == 1 and "Too few arguments: expected 6, got 2" in r.stderr
    if os.path.exists(O.REF_BINARY):
        q = subprocess.run([O.REF_BINARY, "a", "b"], capture_output=True, text=True)
        assert (q.returncode, q.stderr) == (r.returncode, r.stderr)


@pytest.mark.skipif(not os.path.exists(CLI), reason="reference-hosted CLI not built (reference sources absent)")
def test_cli_fails_loudly_without_gpu(scene_dir, tmp_path):
    import subprocess

    r = subprocess.run([CLI, scene_dir("tiny"), "16", "12", "2", str(tmp_path / "o.ppm")], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))  # no device visible, on a GPU machine too
    assert r.returncode == 1 and "rt_gpu_create failed (-2)" in r.stderr
    assert not (tmp_path / "o.ppm").exists()


def test_python_cli_argument_error(capsys):
    from rt_b200 import cli

    assert cli.main(["prog", "x"]) == 1
    assert "Too few arguments: expected 6, got 1" in capsys.readouterr().err
