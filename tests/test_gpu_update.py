"""rt_gpu_update_geometry on the B200: the refit tree reproduces the upload bit for bit on a round trip, stays a valid
tree under large deformations, hits what the float64 brute force hits even with the worst topology, renders what a fresh
upload renders, keeps the handle's state, refuses what it must; and the Python CLI's RT_FRAMES."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

import gen_gltf
import hit_scenarios as hs
from test_gpu_hits import _scenario, view_ids

import rt_b200
from rt_b200 import _abi, cli, gltf, gpu, host

pytestmark = pytest.mark.gpu

STAT_KEYS = ("samples", "extension_rays", "light_pdf_rays", "shades")


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hc():
    return hs.hostcheck()


# ---- deformations --------------------------------------------------------------------------------------------------------
def moved(sc, pos, normals=None):
    """A copy of `sc` with the same triangles at `pos` (and `normals`), its light BVH built over the new positions."""
    s = copy.copy(sc)
    s.tri_pos = np.ascontiguousarray(pos, np.float32).reshape(sc.n_tris, 3, 3)
    if normals is not None:
        s.tri_normals = np.ascontiguousarray(normals, np.float32).reshape(sc.n_tris, 3, 3)
    return gltf.build_light_bvh(s)


def _rot_y(deg):
    a = np.radians(deg)
    return np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])


def rotated(sc, deg, centre=None):
    p = sc.tri_pos.astype(np.float64)
    c = p.reshape(-1, 3).mean(0) if centre is None else np.asarray(centre, np.float64)
    R = _rot_y(deg)
    return moved(sc, (p - c) @ R.T + c, sc.tri_normals.astype(np.float64) @ R.T)


def quarter_turn(sc):
    """(x, y, z) -> (-y, x, z), exactly: every +0 y coordinate (the golden scenes' floors) becomes a -0 x coordinate."""
    p, n = sc.tri_pos, sc.tri_normals
    return moved(sc, np.stack([-p[..., 1], p[..., 0], p[..., 2]], -1), np.stack([-n[..., 1], n[..., 0], n[..., 2]], -1))


def mixed_zeros(sc):
    """every other zero coordinate of `sc` made -0: +0 and -0 meet in the same boxes on the same axis"""
    p = sc.tri_pos.copy()
    z = np.flatnonzero(p == 0)
    p.flat[z[::2]] = -0.0
    return moved(sc, p)


def subset_moved(sc, every=7, shift=(0.3, 0.1, -0.2), deg=25.0):
    """Every `every`-th triangle rotated about its group's centre and translated by `shift` times the scene's extent."""
    p = sc.tri_pos.astype(np.float64).copy()
    sel = np.arange(sc.n_tris) % every == 0
    lo, hi = p.reshape(-1, 3).min(0), p.reshape(-1, 3).max(0)
    c = p[sel].reshape(-1, 3).mean(0)
    p[sel] = (p[sel] - c) @ _rot_y(deg).T + c + np.asarray(shift) * (hi - lo)
    return moved(sc, p)


def deformed(sc, kind):
    if kind == "subset":
        return subset_moved(sc)
    if kind == "rotation":
        return rotated(sc, 37.0)
    if kind == "scale_1e3":
        return moved(sc, sc.tri_pos.astype(np.float64) * 1e3)
    if kind == "translate_3e4":
        return moved(sc, sc.tri_pos.astype(np.float64) + np.array([3e4, -3e4, 3e4]))
    if kind == "teleport":
        perm = np.random.default_rng(5).permutation(sc.n_tris)
        return moved(sc, sc.tri_pos[perm], sc.tri_normals[perm])
    raise ValueError(kind)


def lights_translated(sc, shift=(0.0, -0.15, 0.4)):
    """`sc` with its emissive triangles moved: the light side of an update."""
    em = (sc.materials["emission"][sc.tri_material] != 0).any(axis=1)
    p = sc.tri_pos.astype(np.float64).copy()
    lo, hi = p.reshape(-1, 3).min(0), p.reshape(-1, 3).max(0)
    p[em] += np.asarray(shift) * (hi - lo)
    return moved(sc, p)


# ---- readouts -------------------------------------------------------------------------------------------------------------
def selectors(rt):
    return [rt.debug_bvh(0, np.uint32)] + [rt.debug_bvh(i, np.uint8) for i in (1, 2, 3, 4)]


def links(qn):
    return qn.reshape(-1, 64)[:, 36:52].copy()


def snapshot(rt, w, h, spp=16):
    ids = rt.primary_ids(w, h)
    rt.render(w, h, spp, seed=3)
    img, st = rt.readback()
    return selectors(rt), ids, img, rt.readback_rgb8(), {k: st[k] for k in STAT_KEYS}


def assert_same_snapshot(a, b):
    for i, (x, y) in enumerate(zip(a[0], b[0])):
        assert x.tobytes() == y.tobytes(), f"selector {i}"
    assert np.array_equal(a[1], b[1])
    assert a[2].tobytes() == b[2].tobytes() and a[3].tobytes() == b[3].tobytes()
    assert a[4] == b[4]


def _size(manifest, name):
    m = manifest["scenes"][name]
    return (m["ids_width"], m["ids_height"]) if name == "big_lights" else (m["width"], m["height"])


def _scene(name, golden_scene, big_scene):
    return big_scene if name == "big_lights" else golden_scene(name)


# ---- round trip ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny", "texall", "small_lights", "big_lights"])
def test_round_trip_is_bit_identical(name, rt, manifest, golden_scene, big_scene):
    A = _scene(name, golden_scene, big_scene)
    w, h = _size(manifest, name)
    rt.upload_scene(A)
    ref = snapshot(rt, w, h)
    rt.update_geometry(A)  # straight after the upload: changes nothing
    assert_same_snapshot(snapshot(rt, w, h), ref)
    for B in (rotated(A, 10.0), lights_translated(A) if name != "tiny" else subset_moved(A, every=2)):
        rt.update_geometry(B)
        assert links(rt.debug_bvh(3, np.uint8)).tobytes() == links(ref[0][3]).tobytes()
        rt.update_geometry(A)
        assert_same_snapshot(snapshot(rt, w, h), ref)


@pytest.mark.parametrize("how", ["quarter_turn", "mixed_zeros"])
@pytest.mark.parametrize("name", ["tiny", "small_lights"])
def test_round_trip_with_negative_zeros(name, how, rt, manifest, golden_scene):
    """The golden scenes have +0 coordinates and no -0.  A quarter turn brings -0 in, and mixed_zeros puts +0 and -0 on
    the same axis of the same boxes: the refit must reduce signed zeros as the build does."""
    A = {"quarter_turn": quarter_turn, "mixed_zeros": mixed_zeros}[how](golden_scene(name))
    assert ((A.tri_pos == 0) & np.signbit(A.tri_pos)).any()
    w, h = _size(manifest, name)
    rt.upload_scene(A)
    ref = snapshot(rt, w, h)
    rt.update_geometry(rotated(A, 33.0))
    rt.update_geometry(A)
    assert_same_snapshot(snapshot(rt, w, h), ref)


# ---- refit validity ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,kind", [("small_lights", k) for k in ("subset", "rotation", "scale_1e3", "translate_3e4", "teleport")] +
                         [("big_lights", "subset"), ("big_lights", "teleport")])
def test_refit_tree_is_valid(name, kind, rt, hc, golden_scene, big_scene):
    A = _scene(name, golden_scene, big_scene)
    rt.upload_scene(A)
    info0, qn0 = rt.debug_bvh(0, np.uint32), rt.debug_bvh(3, np.uint8)
    B = deformed(A, kind)
    rt.update_geometry(B)
    info, nodes, objects, qn, tris = (rt.debug_bvh(0, np.uint32), rt.debug_bvh(1, _abi.NODE_DTYPE), rt.debug_bvh(2, np.uint32),
                                      rt.debug_bvh(3, np.uint8), rt.debug_bvh(4, np.uint8))
    hs.check_tree(hc, B, info, nodes, objects, qn, tris)
    assert np.array_equal(info, info0) and links(qn).tobytes() == links(qn0).tobytes()
    t = tris.reshape(-1, 64)[:-1]
    ax = t[:, :12].copy().view(np.float32).reshape(-1, 3)  # DTri: a, then (e1 e2 from byte 16)
    assert np.array_equal(ax, B.tri_pos[objects.astype(np.int64), 0])


# ---- hits against the float64 brute force --------------------------------------------------------------------------------
def _brute_force_run(rt, hc, name, big_scene=None):
    sc, tri, rays, pix, exp = _scenario(name, hc, big_scene)
    if name == "big_lights":
        start = subset_moved(sc, every=5, shift=(0.45, 0.0, -0.3), deg=60.0)
    else:
        start = moved(sc, tri[np.random.default_rng(11).permutation(len(tri))])
    rt.upload_scene(start)  # the tree of another geometry
    rt.update_geometry(sc)
    n_views = len(rays) - (0 if pix is None else len(pix))
    ids = view_ids(rt, rays[:n_views])
    if pix is not None:
        ids = np.concatenate([ids, rt.primary_ids(256, 256).reshape(-1)[pix]])
    bad = exp.wrong(ids)
    print(f"{name} [refit]: {len(rays)} rays, decidable {exp.dec.mean():.3f}, mismatches {int(bad.sum())}")
    assert not bad.any(), f"{name}: {int(bad.sum())} decidable rays miss their nearest hit after a refit"
    assert exp.dec.mean() >= hs.DECIDABLE_FLOOR[name]


@pytest.mark.parametrize("name", sorted(hs.SCENARIOS))
def test_refit_hits_what_the_brute_force_hits(name, rt, hc):
    _brute_force_run(rt, hc, name)


def test_refit_hits_on_the_260k_scene(rt, hc, big_scene):
    _brute_force_run(rt, hc, "big_lights", big_scene)


# ---- against a fresh upload ----------------------------------------------------------------------------------------------
def _compare_with_fresh(rt, A, B, w, h):
    rt.upload_scene(A)
    rt.update_geometry(B)
    ids_u = rt.primary_ids(w, h)
    rt.render(200, 200, 8, seed=5)
    img_u, st_u = rt.readback()
    rt.upload_scene(B)
    ids_f = rt.primary_ids(w, h)
    rt.render(200, 200, 8, seed=5)
    img_f, st_f = rt.readback()
    assert (ids_u == ids_f).mean() >= 0.9999
    rel = np.abs(img_u - img_f) / (np.abs(img_f) + 1e-3)
    assert (rel.max(axis=2) > 1e-3).mean() <= 0.01
    assert abs(st_u["extension_rays"] - st_f["extension_rays"]) <= 1e-3 * st_f["extension_rays"]
    return img_u, img_f


@pytest.mark.parametrize("case", ["small_lights_lights_moved", "small_lights_rotation", "texall_subset", "big_lights_subset"])
def test_update_renders_what_a_fresh_upload_renders(case, rt, manifest, golden_scene, big_scene):
    name, how = {"small_lights_lights_moved": ("small_lights", lights_translated),
                 "small_lights_rotation": ("small_lights", lambda s: rotated(s, 20.0)),
                 "texall_subset": ("texall", subset_moved), "big_lights_subset": ("big_lights", subset_moved)}[case]
    A = _scene(name, golden_scene, big_scene)
    B = how(A)
    w, h = _size(manifest, name)
    img_u, img_f = _compare_with_fresh(rt, A, B, w, h)
    if case == "small_lights_lights_moved":  # the moved emitters changed the image
        rt.upload_scene(A)
        rt.render(200, 200, 8, seed=5)
        assert not np.allclose(rt.readback()[0], img_f, rtol=1e-2, atol=1e-2)


# ---- state and errors ----------------------------------------------------------------------------------------------------
def test_readbacks_survive_an_update(rt, golden_scene):
    A = golden_scene("small_lights")
    rt.upload_scene(A)
    ids = rt.primary_ids(16, 16)
    rt.update_geometry(rotated(A, 15.0))
    ids_moved = np.empty_like(ids)
    assert gpu.lib().rt_gpu_readback(rt._h, None, ids_moved.ctypes.data_as(C.c_void_p), None) == 0
    assert np.array_equal(ids_moved, ids)  # the ids of the last render, not of the moved scene
    rt.render(64, 64, 8, seed=2)
    img, st = rt.readback()
    rgb8 = rt.readback_rgb8()
    ptr = rt.accum_device_ptr()
    rt.update_geometry(A)
    img2, st2 = rt.readback()
    assert img2.tobytes() == img.tobytes() and rt.readback_rgb8().tobytes() == rgb8.tobytes() and st2 == st
    assert rt.accum_device_ptr() == ptr
    assert np.array_equal(rt.primary_ids(16, 16), ids)  # the round-tripped scene
    # accumulation after an update adds samples of the new geometry
    rt.render(32, 32, 8, seed=4, sample_begin=0, sample_end=4)
    rt.update_geometry(rotated(A, 15.0))
    rt.render(32, 32, 8, seed=4, sample_begin=4, sample_end=8, accumulate=True)
    assert rt.stats()["samples"] == 32 * 32 * 4  # stats are the last render's


def test_adaptive_views_and_projected_renders_after_an_update(rt, golden_scene):
    A = golden_scene("small_lights")
    B = rotated(A, 12.0)
    cams = [B.camera(), rt_b200.Camera(B.camera_position + 0.05, B.camera_right, B.camera_up, B.camera_forward, B.fov_x)]
    projs = [rt_b200.Projection.pinhole(), rt_b200.Projection.thin_lens(0.01, 1.0)]
    out = {}
    for fresh in (False, True):
        if fresh:
            rt.upload_scene(B)
        else:
            rt.upload_scene(A)
            rt.update_geometry(B)
        rt.render_adaptive(32, 32, 64, 8, 8, 0.05, seed=1)
        a = rt.readback()[0]
        rt.render_views(cams, 32, 32, 8, seed=1)
        v = rt.readback()[0]
        rt.render_projected(cams, projs, 32, 32, 8, seed=1, adaptive=(8, 8, 0.05))
        p = rt.readback()[0]
        out[fresh] = (a, v, p, rt.primary_ids(32, 32, cameras=cams, projections=projs))
    for x, y in zip(out[False][:3], out[True][:3]):
        assert x.shape == y.shape and np.isfinite(x).all()
        rel = np.abs(x - y) / (np.abs(y) + 1e-3)
        assert (rel.max(axis=-1) > 1e-3).mean() <= 0.01
    assert (out[False][3] == out[True][3]).mean() >= 0.999


def _status(name):
    return next(code for code, n in _abi.STATUS.items() if n == name)


def _call(rt, u):
    return gpu.lib().rt_gpu_update_geometry(rt._h, C.byref(u) if u is not None else None)


def test_refusals_leave_the_scene_untouched(rt, golden_scene):
    A = golden_scene("small_lights")
    rt.upload_scene(A)
    rt.render(48, 48, 4, seed=9)
    ref = rt.readback()[0]
    B = rotated(A, 30.0)
    INVALID = _status("RT_ERR_INVALID_ARG")

    def refused(u):
        assert _call(rt, u) == INVALID, gpu.lib().rt_gpu_last_error()
        rt.render(48, 48, 4, seed=9)
        assert rt.readback()[0].tobytes() == ref.tobytes()

    refused(None)
    u = B.geometry_update()
    u.n_tris = A.n_tris - 1
    refused(u)
    for field in ("tri_pos", "tri_normals"):
        u = B.geometry_update()
        setattr(u, field, None)
        refused(u)
    u = B.geometry_update()  # another number of lights
    u.light_bvh.n_objects -= 1
    refused(u)
    bad_ids = copy.copy(B)
    bad_ids.light_bvh = _abi.BvhData(B.light_bvh.nodes, B.light_bvh.objects.copy(), B.light_bvh.root)
    bad_ids.light_bvh.objects[3] = A.n_tris
    refused(bad_ids.geometry_update())
    bad_links = copy.copy(B)
    nodes = B.light_bvh.nodes.copy()
    nodes[0]["left_child"] = len(nodes) + 5
    bad_links.light_bvh = _abi.BvhData(nodes, B.light_bvh.objects, B.light_bvh.root)
    refused(bad_links.geometry_update())
    u = B.geometry_update()
    u.light_bvh.nodes = None
    refused(u)


@pytest.mark.parametrize("how", ["flag", "RT_HOST_BUILD", "RT_KEEP_HOST_BVH"])
def test_host_built_trees_are_refused(how, rt, golden_scene):
    A = golden_scene("small_lights")
    B = rotated(A, 30.0)
    if how == "flag":
        d = A.desc()
        d.flags = 1  # RT_SCENE_KEEP_HOST_BVH
        assert gpu.lib().rt_gpu_upload_scene(rt._h, C.byref(d)) == 0
    else:
        os.environ[how] = "1"
        try:
            rt.upload_scene(A)
        finally:
            del os.environ[how]
    rt.render(32, 32, 4, seed=1)
    ref = rt.readback()[0]
    assert _call(rt, B.geometry_update()) == _status("RT_ERR_INVALID_ARG")
    assert "device" in gpu.lib().rt_gpu_last_error().decode()
    os.environ["RT_HOST_BUILD"] = "0"  # the upload's record decides, not the environment at update time
    try:
        assert _call(rt, B.geometry_update()) == _status("RT_ERR_INVALID_ARG")
    finally:
        del os.environ["RT_HOST_BUILD"]
    rt.render(32, 32, 4, seed=1)
    assert rt.readback()[0].tobytes() == ref.tobytes()


def test_text_scene_and_no_scene_are_refused(golden_scene):
    B = golden_scene("tiny")
    with gpu.RtGpu(1, 0) as g:
        assert _call(g, B.geometry_update()) == _status("RT_ERR_NO_SCENE")
        from rt_b200 import textscene

        g.upload_text_scene(textscene.TextScene())
        assert _call(g, B.geometry_update()) == _status("RT_ERR_INVALID_ARG")


def test_non_finite_vertex_drops_the_scene(rt, golden_scene):
    A = golden_scene("texall")
    rt.upload_scene(A)
    p = A.tri_pos.copy()
    p[17, 2, 1] = np.nan
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_BAD_SCENE"):
        rt.update_geometry(moved(A, p))
    with pytest.raises(gpu.RtGpuError, match="RT_ERR_NO_SCENE"):
        rt.render(16, 16, 1)
    assert _call(rt, A.geometry_update()) == _status("RT_ERR_NO_SCENE")
    rt.upload_scene(A)  # the next upload brings the handle back
    rt.render(16, 16, 1)


def test_empty_scene_updates(rt):
    sc = hs.triangles_scene(np.zeros((0, 3, 3), np.float32))
    rt.upload_scene(sc)
    rt.update_geometry(sc)
    ids = rt.primary_ids(8, 8)
    assert (ids == -1).all()


def test_tangents_follow_the_update(rt, manifest, golden_scene):
    """DTangent exists only while some tangent differs from (1, 0, 0); the round trip through a tangent-carrying state
    restores the upload."""
    A = golden_scene("texall")
    w, h = _size(manifest, "texall")
    rt.upload_scene(A)
    ref = snapshot(rt, w, h)
    T = copy.copy(A)
    T.tri_tangents = np.tile(np.array([0, 0, 1], np.float32), (A.n_tris, 3, 1))
    rt.update_geometry(T)
    rt.render(w, h, 4, seed=3)
    assert np.isfinite(rt.readback()[0]).all()
    rt.update_geometry(A)
    assert_same_snapshot(snapshot(rt, w, h), ref)


# ---- two devices ---------------------------------------------------------------------------------------------------------
def _n_dev():
    try:
        return gpu.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_dev() < 2, reason="needs >= 2 GPUs")
def test_two_devices_match_one_after_an_update(golden_scene):
    A = golden_scene("small_lights")
    B = lights_translated(rotated(A, 8.0))
    imgs = []
    for n in (1, 2):
        with gpu.RtGpu(n, 0) as g:
            g.upload_scene(A)
            g.update_geometry(B)
            g.render(96, 64, 32, seed=11)
            imgs.append(g.readback()[0])
    assert np.allclose(imgs[1], imgs[0], rtol=2e-6, atol=1e-7)


# ---- CLI -----------------------------------------------------------------------------------------------------------------
def test_cli_frames(tmp_path, monkeypatch):
    g = gen_gltf.tiny()
    g.animation([(0, "translation", [0.0, 1.0], [[0, 0, 0], [0.3, 0.1, -0.4]], "LINEAR"),
                 (1, "translation", [0.0, 1.0], [[0.0, 1.6, 2.5], [0.2, 1.7, 2.3]], "LINEAR")])
    path = g.write(str(tmp_path))
    w, h, spp, seed, fps = 64, 48, 16, 7, 4.0
    for k in ("RT_CAMERAS", "RT_ANIMATION", "RT_ADAPTIVE", "RT_PROJECTION", "RT_ENV_MAP", "RT_GPUS"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("RT_FRAMES", f"3:{fps}")
    monkeypatch.setenv("RT_SEED", str(seed))
    out = tmp_path / "frames" / "anim.ppm"
    assert cli.main(["rt", path, str(w), str(h), str(spp), str(out)]) == 0
    frames = [tmp_path / "frames" / f"anim_{f}.ppm" for f in range(3)]
    assert all(f.exists() for f in frames)
    t0, _ = gltf.animation_range(path)
    for f, frame in enumerate(frames):
        mean, _ = cli.run_raytracer(gltf.load_gltf(path, w / h, time=t0 + f / fps), w, h, spp, seed=seed + f)
        ref = tmp_path / f"ref_{f}.ppm"
        host.write_ppm(str(ref), host.tonemap_rgb8(mean))
        if f == 0:
            assert frame.read_bytes() == ref.read_bytes()
        else:
            a = np.frombuffer(frame.read_bytes()[-w * h * 3:], np.uint8).reshape(h, w, 3).astype(int)
            b = np.frombuffer(ref.read_bytes()[-w * h * 3:], np.uint8).reshape(h, w, 3).astype(int)
            assert (np.abs(a - b).max(axis=2) > 1).mean() <= 0.01
    # the frames differ: the geometry and the camera moved
    assert frames[0].read_bytes() != frames[2].read_bytes()
