"""Closest hits of the host compilation of the traversal (hc_trace_rays: the library's SAH tree through the exact binary
nodes and through the quantised 4-wide nodes in k_extend's arithmetic, closest_hit_q4) against the float64 brute force
hc_brute_hits, on the scenarios of hit_scenarios.py.  No GPU needed: the node tests and the packer are the code the
kernels run, so a box that loses a hit loses it here first."""
import ctypes as C

import numpy as np
import pytest

import hit_scenarios as hs


@pytest.fixture(scope="module")
def hc():
    return hs.hostcheck()


def _trace(hc, sc, rays):
    m = len(rays)
    te, tq = np.zeros(m, np.float32), np.zeros(m, np.float32)
    ie, iq = np.zeros(m, np.int32), np.zeros(m, np.int32)
    d = sc.desc()
    hc.hc_set_rebuild(1)
    try:
        rc = hc.hc_trace_rays(C.byref(d), C.c_uint64(m), hs._ptr(rays), hs._ptr(ie), hs._ptr(te), hs._ptr(iq), hs._ptr(tq))
    finally:
        hc.hc_set_rebuild(0)
    assert rc == 0, rc
    return ie, te, iq, tq


def _report(name, exp, rays, got):
    """Fail with the first few wrong rays of each traversal (expected id and t, returned id and t)."""
    lines, total = [], 0
    for label, (ids, t) in got.items():
        bad = exp.wrong(ids)
        total += int(bad.sum())
        print(f"{name} [{label}]: {len(rays)} rays, decidable {exp.dec.mean():.3f}, mismatches {int(bad.sum())}")
        for i in np.flatnonzero(bad)[:4]:
            lines.append(f"  {label} ray {i} o={rays[i, :3].tolist()} d={rays[i, 3:].tolist()}: expected {exp.k[i]} t={exp.t[i]:.9g} "
                         f"(ties {exp.ties[i]}), got {ids[i]} t={t[i]:.9g}")
    assert total == 0, f"{name}: {total} decidable rays miss their nearest hit\n" + "\n".join(lines)


@pytest.mark.parametrize("name", sorted(hs.SCENARIOS))
def test_host_traversal_hits_what_the_brute_force_hits(name, hc):
    tri, rays = hs.make(name, hs.N_RAYS)
    sc = hs.triangles_scene(tri)
    exp = hs.Expected(hc, tri, rays, sc.eps)
    ie, te, iq, tq = _trace(hc, sc, rays)
    _report(name, exp, rays, {"exact": (ie, te), "q4": (iq, tq)})
    assert exp.dec.mean() >= hs.DECIDABLE_FLOOR[name]
    assert (exp.k[exp.dec] >= 0).mean() > 0.3


def test_host_traversal_on_the_260k_scene(hc, big_scene):
    rays = hs.big_lights_rays(big_scene, hs.BIG_RAYS)
    tri = np.ascontiguousarray(big_scene.tri_pos, np.float32)
    exp = hs.Expected(hc, tri, rays, big_scene.eps)
    ie, te, iq, tq = _trace(hc, big_scene, rays)
    _report("big_lights", exp, rays, {"exact": (ie, te), "q4": (iq, tq)})
    assert exp.dec.mean() >= hs.DECIDABLE_FLOOR["big_lights"]


def test_zero_area_triangles_are_never_hit(hc):
    tri, rays = hs.make("degenerate", hs.N_RAYS)
    zero = np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]).astype(np.float64), axis=1) == 0
    assert zero.sum() == 2000
    sc = hs.triangles_scene(tri)
    ie, _, iq, _ = _trace(hc, sc, rays)
    for ids in (ie, iq):
        assert not zero[ids[ids >= 0]].any()


@pytest.mark.parametrize("name", sorted(hs.SCENARIOS))
def test_brute_force_matches_its_numpy_statement(name, hc):
    """hc_brute_hits against the same rule written in numpy, on 200 rays of each scenario."""
    tri, rays = hs.make(name, hs.N_RAYS)
    rays = rays[np.random.default_rng(1).choice(len(rays), 200, replace=False)]
    exp = hs.Expected(hc, tri, rays, 1e-4)
    k, t, ties, dec = hs.brute_numpy(tri, rays, 1e-4)
    assert np.array_equal(exp.k, k) and np.array_equal(exp.ties, ties) and np.array_equal(exp.dec, dec)
    hit = k >= 0
    assert np.allclose(exp.t[hit], t[hit], rtol=1e-9, atol=0)


def test_brute_force_by_hand():
    """Three rays whose answer is known without any arithmetic doubt: a clear hit of the nearer of two parallel
    triangles, a ray through the shared edge of two triangles (borderline: not decidable), and a clear miss."""
    hc = hs.hostcheck()
    tri = np.array([[[-1, -1, 0], [1, -1, 0], [0, 1, 0]], [[-1, -1, 1], [1, -1, 1], [0, 1, 1]],
                    [[2, 0, 0], [3, 0, 0], [2, 1, 0]], [[3, 0, 0], [3, 1, 0], [2, 1, 0]]], np.float32)
    rays = np.array([[0, 0, 2, 0, 0, -1], [2.5, 0.5, 2, 0, 0, -1], [5, 5, 2, 0, 0, -1]], np.float32)
    exp = hs.Expected(hc, tri, rays, 1e-4)
    assert exp.k.tolist() == [1, -1, -1]
    assert exp.t[0] == 1.0 and exp.ties[0] == 1
    assert exp.dec.tolist() == [True, False, True]
