"""Closest hits of the kernels against the float64 brute force (hc_brute_hits) on the scenarios of hit_scenarios.py.
Arbitrary rays go through the existing C ABI as 1x1-pixel views: at width = height = 1 the pixel centre's camera term
is (0.5 * 2 - 1) * tan = 0 exactly, so view i traces (position_i, normalize(forward_i)) and returns one id.  Each
scenario also renders one ordinary view of the scene camera (k_generate) and checks a sample of its pixels.

Four configurations: the device build, RT_HOST_BUILD=1, RT_KEEP_HOST_BVH=1 with a tree from rt_b200.host.build_bvh,
and librt_gpu_wide8.so (k_extend8) in a child pytest, as in test_eight_wide_build_keeps_parity."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import hit_scenarios as hs
import rt_b200
from rt_b200 import gpu, host

from conftest import ROOT

pytestmark = pytest.mark.gpu

CONFIGS = ["device", "host_build", "keep_host"]
PIXEL_SAMPLE = 4096  # pixels of the 256 x 256 view checked against the brute force


@pytest.fixture(scope="module")
def rt():
    g = gpu.RtGpu(1, 0)
    yield g
    g.close()


@pytest.fixture(scope="module")
def hc():
    return hs.hostcheck()


_expected = {}


def _with_view(sc, tri, rays):
    """Aim the scene camera at the geometry's box; append a sample of its 256 x 256 pixel rays to `rays`."""
    lo, hi = tri.reshape(-1, 3).min(0).astype(np.float64), tri.reshape(-1, 3).max(0).astype(np.float64)
    c, ext = (lo + hi) / 2, max(float((hi - lo).max()), 1e-3)
    pos = (c + ext * np.array([0.3, 0.2, 1.5])).astype(np.float32)
    fwd = hs._unit(c - pos.astype(np.float64))
    right = hs._unit(np.cross(fwd, [0.0, 1.0, 0.0]))
    up = np.cross(right, fwd)
    sc.camera_position, sc.camera_forward = pos, fwd.astype(np.float32)
    sc.camera_right, sc.camera_up = right.astype(np.float32), up.astype(np.float32)
    sc.fov_x = np.float32(1.0)
    w = h = 256
    tx = np.tan(np.float64(sc.fov_x) / 2)
    pix = np.random.default_rng(7).choice(w * h, PIXEL_SAMPLE, replace=False)
    px, py = pix % w + 0.5, pix // w + 0.5
    a, b = (px * 2 / w - 1) * tx, (py * 2 / h - 1) * tx
    d = hs._unit(a[:, None] * right - b[:, None] * up + fwd).astype(np.float32)
    return np.concatenate([rays, np.concatenate([np.repeat(pos[None], len(d), 0), d], 1)]), pix


def _scenario(name, hc, big_scene=None):
    if name not in _expected:
        if name == "big_lights":
            sc = big_scene
            tri = np.ascontiguousarray(sc.tri_pos, np.float32)
            rays, pix = hs.big_lights_rays(sc, hs.BIG_RAYS), None
        else:
            tri, rays = hs.make(name, hs.N_RAYS)
            sc = hs.triangles_scene(tri)
            rays, pix = _with_view(sc, tri, rays)
        _expected[name] = (sc, tri, rays, pix, hs.Expected(hc, tri, rays, sc.eps))
    return _expected[name]


def view_ids(rt, rays):
    """One primary id per ray (n x 6: origin, unit direction) through 1x1-pixel views, 2^16 views per call."""
    out = []
    for s in range(0, len(rays), hs.VIEW_CHUNK):
        cams = [rt_b200.Camera(r[:3], (1, 0, 0), (0, 1, 0), r[3:], 1.0) for r in rays[s:s + hs.VIEW_CHUNK]]
        out.append(rt.primary_ids(1, 1, cameras=cams).reshape(-1))
    return np.concatenate(out) if out else np.zeros(0, np.int32)


def _upload(rt, sc, config):
    env = {"host_build": "RT_HOST_BUILD", "keep_host": "RT_KEEP_HOST_BVH"}.get(config)
    keep = sc.scene_bvh
    if config == "keep_host" and len(sc.scene_bvh.nodes) == 0:
        sc.scene_bvh = host.build_bvh(sc.tri_pos)
    if env:
        os.environ[env] = "1"
    try:
        rt.upload_scene(sc)
    finally:
        if env:
            del os.environ[env]
        sc.scene_bvh = keep


def _run(name, config, rt, hc, big_scene=None):
    sc, tri, rays, pix, exp = _scenario(name, hc, big_scene)
    _upload(rt, sc, config)
    if config == "device" and not os.environ.get("RT_GPU_LIB"):
        info = rt.debug_bvh(0, np.uint32)
        hs.check_tree(hc, sc, info, rt.debug_bvh(1, rt_b200._abi.NODE_DTYPE), rt.debug_bvh(2, np.uint32), rt.debug_bvh(3, np.uint8),
                      rt.debug_bvh(4, np.uint8))
    n_views = len(rays) - (0 if pix is None else len(pix))
    ids = view_ids(rt, rays[:n_views])
    if pix is not None:
        ids = np.concatenate([ids, rt.primary_ids(256, 256).reshape(-1)[pix]])
    bad = exp.wrong(ids)
    print(f"{name} [{config}{' ' + os.path.basename(os.environ['RT_GPU_LIB']) if os.environ.get('RT_GPU_LIB') else ''}]: "
          f"{len(rays)} rays, decidable {exp.dec.mean():.3f}, mismatches {int(bad.sum())}")
    if bad.any():
        i = np.flatnonzero(bad)[:6]
        m = len(i)
        te, tq = np.zeros(m, np.float32), np.zeros(m, np.float32)
        ie, iq = np.zeros(m, np.int32), np.zeros(m, np.int32)
        sub = np.ascontiguousarray(rays[i])
        d = sc.desc()
        hc.hc_set_rebuild(1)
        try:
            hc.hc_trace_rays(C.byref(d), C.c_uint64(m), hs._ptr(sub), hs._ptr(ie), hs._ptr(te), hs._ptr(iq), hs._ptr(tq))
        finally:
            hc.hc_set_rebuild(0)
        t_got = hs.classify(tri[np.maximum(ids[i], 0)], sub, exp.eps)[2]
        lines = [f"  ray {r} o={rays[r, :3].tolist()} d={rays[r, 3:].tolist()}: expected {exp.k[r]} t={exp.t[r]:.9g} (ties {exp.ties[r]}), "
                 f"got {ids[r]} t={t_got[j] if ids[r] >= 0 else np.inf:.9g}; hc_trace_rays exact {ie[j]} t={te[j]:.9g}, q4 {iq[j]} t={tq[j]:.9g}"
                 for j, r in enumerate(i)]
        pytest.fail(f"{name} [{config}]: {int(bad.sum())} decidable rays miss their nearest hit\n" + "\n".join(lines))
    assert exp.dec.mean() >= hs.DECIDABLE_FLOOR[name]
    zero = np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]).astype(np.float64), axis=1) == 0
    assert not zero[ids[ids >= 0]].any(), "a zero-area triangle was returned"


@pytest.mark.parametrize("config", CONFIGS)
@pytest.mark.parametrize("name", sorted(hs.SCENARIOS))
def test_kernel_hits_what_the_brute_force_hits(name, config, rt, hc):
    _run(name, config, rt, hc)


@pytest.mark.parametrize("config", CONFIGS)
def test_kernel_hits_on_the_260k_scene(config, rt, hc, big_scene):
    _run("big_lights", config, rt, hc, big_scene)


@pytest.mark.parametrize("tail", [16, 1024])
def test_deep_chain_reaches_the_depth_budget(tail, rt, hc):
    """hit_scenarios.depth_chain makes the device builder peel one triangle per level until the depth budget
    (depth + ceil(log2 n) + 2 >= 62) switches to position splits: in kb_small's range with tail = 16, in kb_split's
    with tail = 1024.  Without the budget the tree would be deeper than 62 levels; its 4-wide tree needs more than the
    16 stack entries k_extend keeps in shared memory."""
    if os.environ.get("RT_GPU_LIB"):
        pytest.skip("the device build is not part of this library")
    tri = hs.depth_chain(tail)
    sc = hs.triangles_scene(tri)
    rt.upload_scene(sc)
    info = rt.debug_bvh(0, np.uint32)
    hs.check_tree(hc, sc, info, rt.debug_bvh(1, rt_b200._abi.NODE_DTYPE), rt.debug_bvh(2, np.uint32), rt.debug_bvh(3, np.uint8),
                  rt.debug_bvh(4, np.uint8))  # includes depth < 62
    fd = hs.force_depth(len(tri))
    print(f"chain + {tail}: binary depth {info[5]}, stack need {info[4]}, depth budget fires at {fd}")
    assert info[5] >= fd
    assert info[4] > 16


def test_eight_wide_build_hits_what_the_brute_force_hits():
    """The same scenarios through librt_gpu_wide8.so (k_extend8, qgrid) in a fresh interpreter."""
    if os.environ.get("RT_GPU_LIB"):
        pytest.skip("already running an alternative build")
    lib = os.path.join(ROOT, "raytracing-course-hw-public_b200", "librt_gpu_wide8.so")
    env = dict(os.environ, RT_GPU_LIB=lib)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-p", "no:cacheprovider", "-m", "gpu", os.path.abspath(__file__),
                        "-k", "host_build"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-6000:])
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
