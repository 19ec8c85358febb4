"""Closest-hit scenarios with an independent answer: seeded triangle sets built where BVH builders, quantised node
boxes and slab tests go wrong, rays aimed at them, and the float64 brute force of tests/hostcheck (hc_brute_hits)
that says which triangle each ray must hit.  Shared by test_hits_host.py (the host compilation of the traversal)
and test_gpu_hits.py (the kernels).

Ids are compared, not distances.  A ray counts only when it is decidable (see hc_brute_hits): no triangle that the
float32 arithmetic could get either way lies in front of the nearest clear hit.  On a decidable ray the traversal must
return the brute force's triangle, or, when several clear hits tie within their tolerance, one of those."""
import ctypes as C
import os
import zlib

import numpy as np

import rt_b200
from rt_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C_TOL = 16.0  # tolerance factor of hc_brute_hits (<= 2^7): the exact host traversal has no mismatch at this value
VIEW_CHUNK = 1 << 16  # 1x1-pixel views per render_views call


def hostcheck():
    return C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libhostcheck.so"))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def triangles_scene(tri):
    """A SceneData holding only `tri` ([n, 3, 3] float32), no BVH (the library builds it), camera at (0, 0, 5) looking
    down -z."""
    sc = rt_b200.SceneData.load(os.path.join(ROOT, "tests", "golden", "tiny.rtsc"))
    n = len(tri)
    sc.tri_pos = np.asarray(tri, np.float32).reshape(n, 3, 3)
    sc.tri_normals = np.tile(np.array([0, 0, 1], np.float32), (n, 3, 1))
    sc.tri_uv = np.zeros((n, 3, 2), np.float32)
    sc.tri_tangents = None
    sc.tri_material = np.zeros(n, np.uint32)
    sc.scene_bvh = _abi.BvhData(np.zeros(0, _abi.NODE_DTYPE), np.zeros(0, np.uint32), _abi.RT_NO_CHILD)
    sc.light_bvh = _abi.BvhData(np.zeros(0, _abi.NODE_DTYPE), np.zeros(0, np.uint32), _abi.RT_NO_CHILD)
    sc.camera_position = np.array([0, 0, 5], np.float32)
    sc.camera_forward = np.array([0, 0, -1], np.float32)
    sc.camera_right = np.array([1, 0, 0], np.float32)
    sc.camera_up = np.array([0, 1, 0], np.float32)
    return sc


def check_tree(hc, sc, info, nodes, objects, qn, tris):
    """Invariants of a device-built tree downloaded through rt_gpu_debug_get_bvh: every triangle in one leaf, exact
    boxes, the builder's layout, quantised boxes that contain their triangles, and the stack need the upload checked."""
    n = sc.n_tris
    assert info[0] == n and info[6] == 1, info  # built on the device
    assert sorted(objects.tolist()) == list(range(n))
    d = sc.desc()
    out = np.zeros(8)
    rc = hc.hc_tree_stats(C.byref(d), _ptr(nodes), C.c_uint64(len(nodes)), _ptr(objects), C.c_uint64(len(objects)), _ptr(out))
    assert rc == 0, rc
    _, inner, leaves, max_leaf, depth, ok, cost, layout = out
    assert ok == 1.0, "triangle coverage / exact boxes"
    assert layout == 1.0 and inner == leaves - 1 and max_leaf <= 8 and depth == info[5] and depth < 62
    res = np.zeros(4)
    root4 = C.c_int32(int(np.int32(np.uint32(info[3]))))
    rc = hc.hc_wide_containment_arrays(_ptr(qn), C.c_uint64(len(qn) // 64), root4, _ptr(tris), C.c_uint64(len(tris) // 64), _ptr(res))
    assert rc == 0, rc
    assert res[1] == 0 and res[2] == n  # no quantised plane cuts into a triangle below it; every triangle reached once
    assert res[3] == info[4] <= 96  # the traversal-stack need computed on the device is the host's figure
    return cost, depth, inner


# ---- geometry ---------------------------------------------------------------------------------------------------------
def _soup(rng, n, lo_e, hi_e, half=1.0, offset=(0, 0, 0)):
    c = rng.uniform(-half, half, (n, 3))
    e = 10 ** rng.uniform(np.log10(lo_e), np.log10(hi_e), (n, 1))
    v = c[:, None, :] + rng.normal(size=(n, 3, 3)) * e[:, :, None]
    return (v + np.asarray(offset, np.float64)).astype(np.float32)


def _flat(rng, n, z, half=1.0):
    c = rng.uniform(-half, half, (n, 2))
    e = 10 ** rng.uniform(-3, -1, (n, 1))
    v = np.empty((n, 3, 3), np.float32)
    v[:, :, :2] = c[:, None, :] + rng.normal(size=(n, 3, 2)) * e[:, :, None]
    v[:, :, 2] = np.float32(z)
    return v


def _grid(k=128):
    """k x k quads of side 2^-7 on z = 0 (two triangles each), a wall on x = 0.5 and one on y = 0.25 (32 x 32 quads
    each, also on multiples of 2^-7): every vertex and edge lies on a bin or quantisation boundary."""
    def quads(a, b, fix_axis, fix, n):
        i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        i, j = i.ravel(), j.ravel()
        h = 2.0 ** -7
        p = [(i * h, j * h), ((i + 1) * h, j * h), ((i + 1) * h, (j + 1) * h), (i * h, (j + 1) * h)]
        out = np.empty((2 * len(i), 3, 3), np.float64)
        for t, idx in enumerate([(0, 1, 2), (0, 2, 3)]):
            for vtx, q in enumerate(idx):
                out[t::2, vtx, a] = p[q][0]
                out[t::2, vtx, b] = p[q][1]
                out[t::2, vtx, fix_axis] = fix
        return out

    floor = quads(0, 1, 2, 0.0, k)
    wall_x = quads(1, 2, 0, 0.5, 32)
    wall_y = quads(0, 2, 1, 0.25, 32)
    return np.concatenate([floor, wall_x, wall_y]).astype(np.float32)


def _rot(rng, n):
    q = rng.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
                     np.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1),
                     np.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)], 1)


def _about(rng, centre, n, lo, hi):
    """n triangles whose centroid is `centre` (up to float32 rounding), random orientation, size log-uniform."""
    base = rng.normal(size=(n, 3, 3))
    base -= base.mean(axis=1, keepdims=True)
    s = 10 ** rng.uniform(np.log10(lo), np.log10(hi), (n, 1, 1))
    return (np.einsum("nij,nvj->nvi", _rot(rng, n), base) * s + centre).astype(np.float32)


def _comb(n=300, r=0.85):
    i = np.arange(n)
    x = r ** i
    s = 0.3 * x
    v = np.zeros((n, 3, 3))
    v[:, 0] = np.stack([x, -s, -s], 1)
    v[:, 1] = np.stack([x, s, -s], 1)
    v[:, 2] = np.stack([x + 0.5 * s, 0 * s, s], 1)
    return v.astype(np.float32)


def depth_chain(tail, per_axis=21, a=0.5):
    """A chain the SAH builders can only peel one triangle at a time: per axis, 21 triangles in the planes
    axis = 2^(-6i) (box centres (2^(-6i), 0, 0) and the same on y and z), then `tail` copies of one triangle centred at
    the origin.  In every node each axis has exactly one box centre outside the lowest of the 8 or 32 centroid bins, so
    every split candidate peels one triangle: the binary depth grows by one per triangle until the depth budget
    (depth + ceil(log2 n) + 2 >= 62) switches to position splits.  tail = 16 reaches it in kb_small's range (<= 32
    triangles), tail = 1024 in kb_split's."""
    base = np.array([[-a, -a, 0], [a, -a, 0], [0, a, 0]], np.float64)  # box centre (0, 0, 0)
    tri = []
    for ax in range(3):
        for i in range(per_axis):
            v = np.roll(base, ax + 1, axis=1)  # the constant coordinate moves to axis `ax`
            v[:, ax] = 2.0 ** (-6 * i)
            tri.append(v)
    return np.array(tri + [base] * tail, np.float32)


def force_depth(n):
    """The binary depth at which the builders' depth budget fires for a chain of n triangles peeled one per level."""
    return next(d for d in range(n) if d + int(np.ceil(np.log2(max(n - d, 1)))) + 2 >= 62)


def _degenerate(rng, n):
    """Zero-area triangles whose cross product is exactly 0 in any precision: a repeated vertex, three points on a
    line parallel to an axis, or one point three times."""
    p = rng.uniform(-1, 1, (n, 3))
    q = p + rng.normal(size=(n, 3)) * 0.1
    v = np.stack([p, q, q], 1)
    line = np.arange(n) % 3 == 1
    v[line, 1] = p[line]
    v[line, 2] = p[line]
    v[line, 1, 0] += 0.05
    v[line, 2, 0] += 0.1
    point = np.arange(n) % 3 == 2
    v[point] = p[point, None, :]
    return v.astype(np.float32)


# ---- rays -------------------------------------------------------------------------------------------------------------
def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _aim(o, p):
    """float32 rays from o (float32) towards p (float64)."""
    o = np.asarray(o, np.float32)
    d = _unit(p - o.astype(np.float64)).astype(np.float32)
    return np.concatenate([o, d], 1)


def _nondegenerate(tri):
    t = tri.astype(np.float64)
    return np.flatnonzero(np.linalg.norm(np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]), axis=1) > 0)


def targeted(rng, tri, n, dist_lo, dist_hi, dirs=None):
    """Rays at interior points of random triangles, every barycentric >= 0.05, from dist_lo..dist_hi away."""
    k = rng.choice(_nondegenerate(tri), n)
    b = rng.dirichlet((1, 1, 1), n) * 0.85 + 0.05
    p = np.einsum("nv,nvi->ni", b, tri[k].astype(np.float64))
    d = _unit(rng.normal(size=(n, 3))) if dirs is None else dirs
    return _aim(p - d * rng.uniform(dist_lo, dist_hi, (n, 1)), p)


def beside(rng, tri, n, dist_lo, dist_hi):
    """Rays aimed just outside an edge (by 1e-6..1e-2 of the edge's length, in the triangle's plane)."""
    k = rng.choice(_nondegenerate(tri), n)
    t = tri[k].astype(np.float64)
    e = rng.integers(0, 3, n)
    a, b, c = t[np.arange(n), e], t[np.arange(n), (e + 1) % 3], t[np.arange(n), (e + 2) % 3]
    p = a + (b - a) * rng.uniform(0.1, 0.9, (n, 1))
    nrm = np.cross(b - a, c - a)
    out = _unit(np.cross(b - a, nrm))  # in-plane, away from c
    out *= np.sign(np.einsum("ni,ni->n", out, a - c))[:, None]
    p += out * np.linalg.norm(b - a, axis=1, keepdims=True) * 10 ** rng.uniform(-6, -2, (n, 1))
    d = _unit(rng.normal(size=(n, 3)))
    return _aim(p - d * rng.uniform(dist_lo, dist_hi, (n, 1)), p)


def random_rays(rng, lo, hi, n):
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    return np.concatenate([o, _unit(rng.normal(size=(n, 3))).astype(np.float32)], 1)


def axis_rays(rng, o):
    """Each origin with one of the six axis directions (exact zeros: 1/d = +-inf in the slab tests)."""
    o = np.asarray(o, np.float32)
    d = np.zeros((len(o), 3), np.float32)
    ax = rng.integers(0, 3, len(o))
    d[np.arange(len(o)), ax] = rng.choice(np.array([-1, 1], np.float32), len(o))
    return np.concatenate([o, d], 1)


def in_plane(rng, n, z, lo, hi, grazing):
    """Rays in the plane z (origin on it or one ulp above, d_z = 0) and, when `grazing`, rays at 1e-4..1e-2 rad
    through it from above and below."""
    z = np.float32(z)
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    o[:, 2] = z
    o[1::2, 2] = np.nextafter(z, np.float32(np.inf))
    d = np.zeros((n, 3))
    d[:, :2] = _unit(rng.normal(size=(n, 2)))
    rays = [np.concatenate([o, d.astype(np.float32)], 1)]
    if grazing:
        p = rng.uniform(lo, hi, (n, 3))
        p[:, 2] = z
        ang = 10 ** rng.uniform(-4, -2, n) * rng.choice([-1, 1], n)
        g = d * np.cos(ang)[:, None]
        g[:, 2] = np.sin(ang)
        rays.append(_aim(p - g * rng.uniform(0.1, 1.0, (n, 1)), p))
    return np.concatenate(rays)


# ---- scenarios --------------------------------------------------------------------------------------------------------
def _mix(rng, tri, n, lo, hi, dist):
    """The common families: targeted, beside, random, axis-parallel."""
    q = n // 4
    return np.concatenate([targeted(rng, tri, q, dist[0], dist[1]), beside(rng, tri, q, dist[0], dist[1]),
                           random_rays(rng, lo, hi, q), axis_rays(rng, rng.uniform(lo, hi, (n - 3 * q, 3)))])


def _soup_scene(rng, n_rays):
    tri = _soup(rng, 40000, 1e-3, 0.3)
    return tri, _mix(rng, tri, n_rays, -1.2, 1.2, (0.05, 1.0))


def _clusters_scene(rng, n_rays):
    centres = rng.uniform(-1, 1, (60, 3))
    small = np.concatenate([_soup(rng, 300, 1e-4, 1e-2, half=0.02, offset=c) for c in centres])
    big = _soup(rng, 32, 0.6, 1.5)
    tri = np.concatenate([small, big])
    return tri, _mix(rng, tri, n_rays, -1.2, 1.2, (0.01, 0.5))


def _scales_scene(rng, n_rays):
    tri = _soup(rng, 20000, 1e-5, 10.0)
    return tri, _mix(rng, tri, n_rays, -2, 2, (1e-4, 1.0))


def _far_scene(offset, half):
    def make(rng, n_rays):
        tri = _soup(rng, 4000, 1e-3 * half, 0.3 * half, half=half, offset=offset)
        o = np.asarray(offset, np.float64)
        q = n_rays // 2
        rays = np.concatenate([targeted(rng, tri, q, 0.5 * half, 3 * half), beside(rng, tri, n_rays // 4, 0.5 * half, 3 * half),
                               axis_rays(rng, o + rng.uniform(-1.2 * half, 1.2 * half, (n_rays - q - n_rays // 4, 3)))])
        return tri, rays
    return make


def _flat_scene(rng, n_rays):
    z = 0.25
    tri = np.concatenate([_flat(rng, 30000, z), _flat(rng, 5000, np.float32(z + 2.0 ** -20))])
    q = n_rays // 4
    rays = np.concatenate([targeted(rng, tri, q, 0.01, 1.0), beside(rng, tri, q, 0.01, 1.0), in_plane(rng, q // 2, z, -1, 1, True),
                           axis_rays(rng, np.c_[rng.uniform(-1, 1, (n_rays - 3 * q, 2)), np.full(n_rays - 3 * q, z)])])
    return tri, rays


def _grid_scene(rng, n_rays):
    tri = _grid()
    h = 2.0 ** -7
    q = n_rays // 4
    # origins on grid planes: every coordinate a multiple of 2^-7 or halfway between two
    o = rng.integers(-8, 136, (n_rays - 3 * q, 3)) * h
    o[::2] += rng.integers(0, 2, (len(o[::2]), 3)) * (h / 2)
    rays = np.concatenate([targeted(rng, tri, q, 0.01, 1.0), beside(rng, tri, q, 0.01, 1.0), in_plane(rng, q // 2, 0.0, 0, 1, True),
                           axis_rays(rng, o)])
    return tri, rays


def _coincident_scene(rng, n_rays):
    one = _about(rng, np.zeros(3), 600, 1e-3, 0.5)
    groups = np.concatenate([_about(rng, c, 20, 1e-3, 0.05) for c in rng.uniform(-1, 1, (40, 3))])
    tri = np.concatenate([one, groups])
    tri = np.concatenate([tri, tri[rng.choice(len(tri), 50, replace=False)]])  # exact duplicates
    return tri, _mix(rng, tri, n_rays, -1.2, 1.2, (0.01, 1.0))


def _comb_scene(rng, n_rays):
    tri = _comb()
    q = n_rays // 2
    down_x = np.c_[np.full(n_rays - q, 2.0), rng.uniform(-0.05, 0.05, (n_rays - q, 2)) * 1e-3]
    rays = np.concatenate([targeted(rng, tri, q, 1e-3, 0.3), _aim(down_x.astype(np.float32), np.c_[np.zeros(len(down_x)), down_x[:, 1:]])])
    return tri, rays


def _chain_scene(rng, n_rays):
    tri = depth_chain(16)
    return tri, _mix(rng, tri, n_rays, -0.6, 1.2, (0.01, 1.0))


def _degenerate_scene(rng, n_rays):
    tri = np.concatenate([_soup(rng, 10000, 1e-3, 0.3), _degenerate(rng, 2000)])
    rng.shuffle(tri)
    return tri, _mix(rng, tri, n_rays, -1.2, 1.2, (0.05, 1.0))


SCENARIOS = {
    "soup": _soup_scene,
    "clusters": _clusters_scene,
    "scales": _scales_scene,
    "far_control": _far_scene((0.0, 0.0, 0.0), 0.05),
    "far_3e3": _far_scene((3e3, 0.0, 0.0), 0.05),
    "far_3e4": _far_scene((3e4, -1e4, 5e3), 0.1),
    "flat": _flat_scene,
    "grid": _grid_scene,
    "coincident": _coincident_scene,
    "comb": _comb_scene,
    "chain": _chain_scene,
    "degenerate": _degenerate_scene,
}

# smallest decidable share each scenario's rays keep (the tests print the measured share; the floors sit below the lowest
# share seen over seeds 0-2, so that a reference gone vacuous fails, not a reseeded scenario)
DECIDABLE_FLOOR = {
    "soup": 0.8, "clusters": 0.75, "scales": 0.8, "far_control": 0.8, "far_3e3": 0.8, "far_3e4": 0.8, "flat": 0.6, "grid": 0.6,
    "coincident": 0.8, "comb": 0.5, "chain": 0.8, "degenerate": 0.8, "big_lights": 0.65,
}
N_RAYS = 24000  # per scenario; big_lights (260k triangles) takes BIG_RAYS
BIG_RAYS = 6000


def make(name, n_rays, seed=0):
    """(triangles [n, 3, 3] float32, rays [m, 6] float32) of a scenario."""
    rng = np.random.default_rng([seed, zlib.crc32(name.encode())])  # a scenario's geometry does not depend on the others
    tri, rays = SCENARIOS[name](rng, n_rays)
    return np.ascontiguousarray(tri, np.float32), np.ascontiguousarray(rays, np.float32)


def big_lights_rays(sc, n_rays, seed=0):
    """Rays inside the 260k-triangle room: targeted at its triangles from inside the room's box, and random."""
    rng = np.random.default_rng([seed, 99])
    tri = sc.tri_pos
    lo, hi = tri.reshape(-1, 3).min(0), tri.reshape(-1, 3).max(0)
    q = n_rays // 2
    p_k = rng.choice(_nondegenerate(tri), q)
    b = rng.dirichlet((1, 1, 1), q) * 0.85 + 0.05
    p = np.einsum("nv,nvi->ni", b, tri[p_k].astype(np.float64))
    o = rng.uniform(lo + 0.1 * (hi - lo), hi - 0.1 * (hi - lo), (q, 3))
    rays = np.concatenate([_aim(o, p), random_rays(rng, lo + 0.1 * (hi - lo), hi - 0.1 * (hi - lo), n_rays - q)])
    return np.ascontiguousarray(rays, np.float32)


# ---- the reference ----------------------------------------------------------------------------------------------------
class Expected:
    """hc_brute_hits over one scenario: k_star, t_star, ties, decidable per ray."""

    def __init__(self, hc, tri, rays, eps):
        n = len(rays)
        self.tri, self.rays, self.eps = tri, rays, float(eps)
        self.k = np.zeros(n, np.int32)
        self.t = np.zeros(n, np.float64)
        self.ties = np.zeros(n, np.int32)
        self.dec = np.zeros(n, np.uint8)
        rc = hc.hc_brute_hits(_ptr(tri), C.c_uint64(len(tri)), _ptr(rays), C.c_uint64(n), C.c_double(self.eps), C.c_double(C_TOL),
                              _ptr(self.k), _ptr(self.t), _ptr(self.ties), _ptr(self.dec))
        assert rc == 0, rc
        self.dec = self.dec.astype(bool)

    def wrong(self, ids):
        """Decidable rays whose id is not acceptable: neither k_star nor, when the nearest clear hits tie, one of them."""
        ids = np.asarray(ids).reshape(-1)
        bad = self.dec & (ids != self.k)
        tie = bad & (self.ties > 1) & (ids >= 0)
        if tie.any():
            i = np.flatnonzero(tie)
            clear, _, t, w = classify(self.tri[ids[i]], self.rays[i], self.eps)
            w_star = classify(self.tri[self.k[i]], self.rays[i], self.eps)[3]
            bad[i[clear & (np.abs(t - self.t[i]) <= w + w_star)]] = False
        return bad


def classify(tri, rays, eps, c_tol=C_TOL):
    """numpy statement of hc_brute_hits' pair rule for the pairs (tri[i], rays[i]): (clear hit, borderline, t, w).  Used
    to accept tie ids and to cross-check the C++ brute force."""
    T = tri.astype(np.float64)
    o, d = rays[:, :3].astype(np.float64), rays[:, 3:].astype(np.float64)
    a, e1, e2 = T[:, 0], T[:, 1] - T[:, 0], T[:, 2] - T[:, 0]
    n = np.cross(e1, e2)
    area2 = np.linalg.norm(n, axis=1)
    with np.errstate(all="ignore"):
        det = -np.einsum("ni,ni->n", d, n)
        y = o - a
        r = np.cross(d, y)
        b = -np.einsum("ni,ni->n", e2, r) / det
        g = np.einsum("ni,ni->n", e1, r) / det
        t = np.einsum("ni,ni->n", y, n) / det
        edges = np.stack([np.linalg.norm(T[:, 2] - T[:, 1], axis=1), np.linalg.norm(e2, axis=1), np.linalg.norm(e1, axis=1)], 1)
        alt = np.where(edges > 0, area2[:, None] / edges, 0.0)
        dist = (np.stack([1 - b - g, b, g], 1) * alt).min(1)
        cosg = np.abs(det) / (np.linalg.norm(d, axis=1) * area2)
        w = c_tol * 2.0 ** -23 * (np.abs(T - o[:, None, :]).max(axis=(1, 2)) + np.abs(t)) / cosg
    ok = (det != 0) & (area2 > 0)
    clear = ok & (dist > w) & (t > eps + w) & (cosg > 1e-4)
    border = ok & ~clear & ~((dist < -w) | (t < eps - w))
    return clear, border, t, w


def brute_numpy(tri, rays, eps, c_tol=C_TOL):
    """The whole of hc_brute_hits in numpy, ray by ray (slow: for a few hundred rays)."""
    n = len(rays)
    k_star, t_star = np.full(n, -1, np.int32), np.full(n, np.inf)
    ties, dec = np.zeros(n, np.int32), np.zeros(n, bool)
    for i in range(n):
        rr = np.repeat(rays[i:i + 1], len(tri), 0)
        clear, border, t, w = classify(tri, rr, eps, c_tol)
        if clear.any():
            j = np.flatnonzero(clear)[np.argmin(t[clear])]
            k_star[i], t_star[i] = j, t[j]
            ties[i] = int((clear & (np.abs(t - t[j]) <= w + w[j])).sum())
            with np.errstate(invalid="ignore"):
                dec[i] = not (border & (t - w < t[j] + w[j])).any()
        else:
            dec[i] = not border.any()
    return k_star, t_star, ties, dec
