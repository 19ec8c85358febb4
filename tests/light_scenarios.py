"""Light-pdf scenarios with an independent answer: seeded scenes whose emissive triangles sit where the light box, the
light BVH's quantised nodes and the light traversal's triangle test go wrong, rays aimed at them, and the float64 brute
force of tests/hostcheck (hc_brute_light_pdf) that bounds each ray's light pdf.  Shared by test_light_pdf_host.py (the
host compilation of light_pdf / light_pdf_q8) and test_gpu_light_pdf.py (k_shade's light-box test + k_lightpdf_list, and
k_extend8's light mode).

The light pdf of a ray is bvh_mix_dist::pdf: over every light triangle the ray meets at t >= eps, both faces, occluded
or not, the sum of |y - x|^2 / (|cos| * area), divided by n_lights.  Every other triangle of a scene is an occluder and
must not change it.  The geometry generators and ray families are those of hit_scenarios.py."""
import ctypes as C
import zlib

import numpy as np

import hit_scenarios as hs
from rt_b200 import gltf

C_TOL = hs.C_TOL  # the pair rule's tolerance factor, also the factor of the per-term tolerance (hc_brute_light_pdf)
N_RAYS = 12000  # per scenario
GLTF_RAYS = 6000  # small_manylights and big_lights


def light_scene(tri, light):
    """A SceneData of `tri` whose triangles `light` (bool mask) carry one appended emissive material; the others keep
    the non-emissive material 0.  Its light BVH is built by gltf.build_light_bvh, the reference's builder."""
    sc = hs.triangles_scene(tri)
    mats = sc.materials[:1].copy()
    mats["emission"] = 0.0
    em = mats.copy()
    em["emission"] = 4.0
    sc.materials = np.concatenate([mats, em])
    sc.tri_material = np.where(np.asarray(light, bool), 1, 0).astype(np.uint32)
    return gltf.build_light_bvh(sc)


def light_tris(sc):
    """The light triangles in the light BVH's object order (n_lights of them, zero-area ones included)."""
    return np.ascontiguousarray(sc.tri_pos[sc.light_bvh.objects], np.float32)


# ---- rays -------------------------------------------------------------------------------------------------------------
def signed_zero_axis(rng, o):
    """axis_rays with every zero direction component made -0.0 on half of the rays (1/d = -inf in the slab tests)."""
    r = hs.axis_rays(rng, o)
    neg = np.zeros(len(r), bool)
    neg[::2] = True
    d = r[:, 3:]
    d[neg[:, None] & (d == 0)] = np.float32(-0.0)
    return r


def from_surface(rng, tri, n):
    """Rays that start on a triangle (an interior point, rounded to float32) and leave in a random direction: every
    bounce off an emitter.  The own triangle sits at t ~ 0 and must not count."""
    k = rng.choice(hs._nondegenerate(tri), n)
    b = rng.dirichlet((1, 1, 1), n) * 0.85 + 0.05
    o = np.einsum("nv,nvi->ni", b, tri[k].astype(np.float64)).astype(np.float32)
    return np.concatenate([o, hs._unit(rng.normal(size=(n, 3))).astype(np.float32)], 1)


def _mix(rng, lights, n, lo, hi, dist):
    """targeted and beside (at the lights), random, axis-parallel with signed zeros"""
    q = n // 4
    return np.concatenate([hs.targeted(rng, lights, q, dist[0], dist[1]), hs.beside(rng, lights, q, dist[0], dist[1]),
                           hs.random_rays(rng, lo, hi, q), signed_zero_axis(rng, rng.uniform(lo, hi, (n - 3 * q, 3)))])


# ---- scenarios: (triangles, light mask, rays) ---------------------------------------------------------------------------
def _ceiling(rng, n_rays):
    """quads of an 8 x 8 grid on the ceiling y = 1 over [-1, 1]^2 as lights, every fifth left out (a ray through the
    hole is inside the light box and meets no light), a soup of occluders below: rays from below (up through the room)
    and from behind (above the ceiling, down)."""
    g = np.linspace(-1, 1, 9)
    quads = []
    for i in range(8):
        for j in range(8):
            if (i + 2 * j) % 5 == 2:
                continue
            a, b, c, d = (g[i], g[j]), (g[i + 1], g[j]), (g[i + 1], g[j + 1]), (g[i], g[j + 1])
            quads += [[a, b, c], [a, c, d]]
    xz = np.array(quads)
    lights = np.stack([xz[..., 0], np.ones(xz.shape[:2]), xz[..., 1]], -1).astype(np.float32)
    occ = hs._soup(rng, 3000, 1e-3, 0.2, half=0.9)
    q = n_rays // 6
    up = hs._unit(rng.normal(size=(q, 3)) * [1, 0, 1] + [0, 1.5, 0])
    down = up * [1, -1, 1]
    rays = np.concatenate([hs.targeted(rng, lights, q, 0.05, 2.0, dirs=up), hs.targeted(rng, lights, q, 0.05, 1.0, dirs=down),
                           hs.beside(rng, lights, q, 0.05, 2.0), hs.random_rays(rng, -1.5, 1.5, q),
                           signed_zero_axis(rng, rng.uniform(-1.5, 1.5, (q, 3))), from_surface(rng, lights, n_rays - 5 * q)])
    return np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)], rays


def _flat(z):
    """3000 lights in the plane z (flat in one axis: at z = 0 the light box's margin on z is 1e-7), occluders around:
    targeted, beside, in-plane and grazing rays, axis-parallel rays from the plane."""
    def make(rng, n_rays):
        lights = hs._flat(rng, 3000, z)
        occ = hs._soup(rng, 2000, 1e-3, 0.1, offset=(0, 0, z))
        q = n_rays // 5
        o = np.c_[rng.uniform(-1, 1, (q, 2)), np.full(q, z)]
        rays = np.concatenate([hs.targeted(rng, lights, q, 0.01, 1.0), hs.beside(rng, lights, q, 0.01, 1.0),
                               hs.in_plane(rng, q // 2, z, -1, 1, True), signed_zero_axis(rng, o),
                               hs.random_rays(rng, -1.2, 1.2, n_rays - 4 * q) + np.r_[0, 0, z, 0, 0, 0].astype(np.float32)])
        return np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)], rays
    return make


def _far(offset, half):
    """hit_scenarios' far soups, every other triangle a light"""
    def make(rng, n_rays):
        tri, rays = hs._far_scene(offset, half)(rng, n_rays)
        light = np.arange(len(tri)) % 2 == 0
        q = n_rays // 6
        o = np.asarray(offset, np.float64)
        away = hs._unit(rng.normal(size=(q // 4, 3)))  # from 10 away, outwards: beyond the light box's margin (3 at 3e4)
        extra = np.concatenate([hs.random_rays(rng, -1.5 * half, 1.5 * half, q - len(away)) + np.r_[o, 0, 0, 0].astype(np.float32),
                                np.c_[o + 10 * away, away].astype(np.float32), from_surface(rng, tri[light], q)])
        return tri, light, np.concatenate([rays[:n_rays - 2 * q], extra])
    return make


def _layers(rng, n_rays):
    """40 light layers 2^-20 apart (two triangles each, every layer turned by its own angle about z), occluders beside
    them: a ray through the stack crosses dozens of lights."""
    z0 = np.float32(0.25)
    tris = []
    for k in range(40):
        a = rng.uniform(0, np.pi)
        c, s = np.cos(a), np.sin(a)
        sq = np.array([[-1, -1], [1, -1], [1, 1], [-1, 1]], np.float64) @ np.array([[c, s], [-s, c]])
        z = np.float64(z0) + k * 2.0 ** -20
        for idx in ((0, 1, 2), (0, 2, 3)):
            tris.append(np.c_[sq[list(idx)], np.full(3, z)])
    lights = np.array(tris, np.float32)
    occ = hs._soup(rng, 1000, 1e-3, 0.1, offset=(0, 0, -0.5))
    q = n_rays // 4
    steep = hs._unit(rng.normal(size=(q, 3)) * [0.5, 0.5, 1])
    rays = np.concatenate([hs.targeted(rng, lights, q, 0.05, 1.0, dirs=steep), hs.targeted(rng, lights, q, 0.05, 1.0),
                           hs.in_plane(rng, q // 2, z0 + np.float32(2.0 ** -15), -1, 1, True),
                           signed_zero_axis(rng, np.c_[rng.uniform(-1.2, 1.2, (n_rays - 3 * q, 2)), rng.uniform(-0.5, 1.0, n_rays - 3 * q)])])
    return np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)], rays


def _duplicates(rng, n_rays):
    """coincident duplicate lights (exact copies of 300 of 1500): a ray through one crosses both, and both count"""
    soup = hs._soup(rng, 1500, 1e-3, 0.3)
    lights = np.concatenate([soup, soup[rng.choice(len(soup), 300, replace=False)]])
    occ = hs._soup(rng, 1500, 1e-3, 0.3)
    return (np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)],
            _mix(rng, lights, n_rays, -1.2, 1.2, (0.05, 1.0)))


def _tiny_under_huge(rng, n_rays):
    """clusters of tiny lights (1e-5 .. 1e-2) under one huge light (z = 0.9, extent 20): rays from above cross both"""
    centres = rng.uniform(-1, 1, (40, 3)) * [1, 1, 0.5]
    tiny = np.concatenate([hs._soup(rng, 100, 1e-5, 1e-2, half=0.02, offset=c) for c in centres])
    huge = np.array([[[-10, -10, 0.9], [10, -10, 0.9], [0, 12, 0.9]]], np.float32)
    lights = np.concatenate([tiny, huge])
    occ = hs._soup(rng, 500, 1e-3, 0.1)
    q = n_rays // 4
    down = hs._unit(rng.normal(size=(q, 3)) * [0.3, 0.3, 0] + [0, 0, -1])
    rays = np.concatenate([hs.targeted(rng, tiny, q, 1.0, 2.5, dirs=down), hs.targeted(rng, tiny, q, 0.01, 0.5),
                           hs.beside(rng, tiny, q, 0.01, 0.5), signed_zero_axis(rng, rng.uniform(-1.2, 1.2, (n_rays - 3 * q, 3)))])
    return np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)], rays


def _chain(rng, n_rays):
    """hit_scenarios.depth_chain as lights: the light BVH the SAH builder makes of it is as deep as it gets"""
    lights = hs.depth_chain(16)
    return lights, np.ones(len(lights), bool), _mix(rng, lights, n_rays, -0.6, 1.2, (0.01, 1.0))


def _zero_area(rng, n_rays):
    """a soup of lights with 500 zero-area lights among them: they never contribute, but they count in n_lights"""
    lights = np.concatenate([hs._soup(rng, 2000, 1e-3, 0.3), hs._degenerate(rng, 500)])
    rng.shuffle(lights)
    occ = hs._soup(rng, 1000, 1e-3, 0.3)
    return (np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)],
            _mix(rng, lights, n_rays, -1.2, 1.2, (0.05, 1.0)))


def _on_lights(rng, n_rays):
    """rays that start on a light triangle of a soup (many meet no other light: their pdf must be exactly 0)"""
    lights = hs._soup(rng, 2000, 1e-3, 0.3)
    occ = hs._soup(rng, 1000, 1e-3, 0.3)
    return np.concatenate([lights, occ]), np.r_[np.ones(len(lights), bool), np.zeros(len(occ), bool)], from_surface(rng, lights, n_rays)


SCENARIOS = {
    "ceiling": _ceiling,
    "flat_z0": _flat(0.0),
    "flat_z3e4": _flat(3e4),
    "far_control": _far((0.0, 0.0, 0.0), 0.05),
    "far_3e3": _far((3e3, 0.0, 0.0), 0.05),
    "far_3e4": _far((3e4, -1e4, 5e3), 0.1),
    "layers": _layers,
    "duplicates": _duplicates,
    "tiny_under_huge": _tiny_under_huge,
    "chain": _chain,
    "zero_area": _zero_area,
    "on_lights": _on_lights,
}
GLTF_SCENES = ["small_manylights", "big_lights"]
# scenarios whose rays must fall in all three box categories: missing the box of all lights, inside it without a light
# hit, and with a clear light hit
BOX_SCENARIOS = {"ceiling", "flat_z0", "flat_z3e4", "far_control", "far_3e3", "far_3e4", "tiny_under_huge"}

# smallest share of "tight" rays (clear light hits, no borderline pair) each scenario keeps (the tests print the
# measured share; the floors sit below the lowest share seen over seeds 0-2, so that a reference gone vacuous fails,
# not a reseeded scenario)
TIGHT_FLOOR = {
    "ceiling": 0.25, "flat_z0": 0.2, "flat_z3e4": 0.2, "far_control": 0.2, "far_3e3": 0.2, "far_3e4": 0.2, "layers": 0.3,
    "duplicates": 0.2, "tiny_under_huge": 0.3, "chain": 0.2, "zero_area": 0.2, "on_lights": 0.02,
    "small_manylights": 0.2, "big_lights": 0.2,
}


def make(name, n_rays=N_RAYS, seed=0):
    """(SceneData, rays [m, 6] float32) of a scenario."""
    rng = np.random.default_rng([seed, zlib.crc32(("light:" + name).encode())])
    tri, light, rays = SCENARIOS[name](rng, n_rays)
    sc = light_scene(np.ascontiguousarray(tri, np.float32), light)
    return sc, np.ascontiguousarray(rays, np.float32)


def gltf_rays(sc, n_rays, seed=0):
    """Rays from inside a glTF room: aimed at its lights, random, axis-parallel with signed zeros."""
    rng = np.random.default_rng([seed, 77])
    lights = light_tris(sc)
    p = sc.tri_pos.reshape(-1, 3)
    lo, hi = p.min(0).astype(np.float64), p.max(0).astype(np.float64)
    lo, hi = lo + 0.1 * (hi - lo), hi - 0.1 * (hi - lo)
    q = n_rays // 3
    k = rng.choice(hs._nondegenerate(lights), q)
    b = rng.dirichlet((1, 1, 1), q) * 0.85 + 0.05
    aim = np.einsum("nv,nvi->ni", b, lights[k].astype(np.float64))
    rays = np.concatenate([hs._aim(rng.uniform(lo, hi, (q, 3)), aim), hs.random_rays(rng, lo, hi, q),
                           signed_zero_axis(rng, rng.uniform(lo, hi, (n_rays - 2 * q, 3)))])
    return np.ascontiguousarray(rays, np.float32)


# ---- the reference ----------------------------------------------------------------------------------------------------
class Bounds:
    """hc_brute_light_pdf over one scene: lo, hi, n_clear, n_border per ray."""

    def __init__(self, hc, sc, rays):
        n = len(rays)
        self.rays = rays
        self.lights = light_tris(sc)
        self.eps = float(sc.eps)
        self.lo, self.hi = np.zeros(n), np.zeros(n)
        self.n_clear, self.n_border = np.zeros(n, np.int32), np.zeros(n, np.int32)
        rc = hc.hc_brute_light_pdf(hs._ptr(self.lights), C.c_uint64(len(self.lights)), hs._ptr(rays), C.c_uint64(n), C.c_double(self.eps),
                                   C.c_double(C_TOL), hs._ptr(self.lo), hs._ptr(self.hi), hs._ptr(self.n_clear), hs._ptr(self.n_border))
        assert rc == 0, rc

    @property
    def tight(self):
        return (self.n_clear > 0) & (self.n_border == 0)

    def wrong(self, pdf):
        """Rays whose pdf is outside [lo, hi], or not exactly 0 without any clear or borderline pair."""
        pdf = np.asarray(pdf, np.float64)
        empty = (self.n_clear == 0) & (self.n_border == 0)
        with np.errstate(invalid="ignore"):
            out = ~((self.lo <= pdf) & (pdf <= self.hi))
        return out | (empty & (pdf != 0.0))

    def report(self, label, pdf, limit=8):
        """Fail text: the first wrong rays with their interval, the value got and n_clear / n_border."""
        bad = np.flatnonzero(self.wrong(pdf))
        lines = [f"{label}: {len(bad)} of {len(pdf)} rays outside their bounds"]
        for i in bad[:limit]:
            lines.append(f"  ray {i} o={self.rays[i, :3].tolist()} d={self.rays[i, 3:].tolist()}: expected [{self.lo[i]:.9g}, {self.hi[i]:.9g}] "
                         f"(clear {self.n_clear[i]}, borderline {self.n_border[i]}), got {pdf[i]:.9g}")
        return "\n".join(lines)


def box_categories(sc, rays):
    """(misses the box of all lights, inside that box without any light pair, -) as bool masks, in float64 on the exact
    box of the light triangles: a miss is a ray whose t >= eps part misses the box grown by twice the upload's margin."""
    lt = light_tris(sc).reshape(-1, 3).astype(np.float64)
    lo, hi = lt.min(0), lt.max(0)
    m = 1e-4 * np.maximum.reduce([hi - lo, np.abs(lo), np.abs(hi), np.full(3, 1e-3)])

    def meets(blo, bhi):
        o, d = rays[:, :3].astype(np.float64), rays[:, 3:].astype(np.float64)
        with np.errstate(all="ignore"):
            inv = 1.0 / d
            a, b = (blo - o) * inv, (bhi - o) * inv
            t0 = np.fmax(np.nanmax(np.fmin(a, b), axis=1), float(sc.eps))
            t1 = np.nanmin(np.fmax(a, b), axis=1)
        return t0 <= t1

    return ~meets(lo - 2 * m, hi + 2 * m), meets(lo, hi)


def bounds_numpy(lights, rays, eps, c_tol=C_TOL):
    """The whole of hc_brute_light_pdf in numpy, ray by ray (slow: for a few hundred rays): (lo, hi, n_clear, n_border)."""
    n, u = len(rays), 2.0 ** -23
    lo, hi = np.zeros(n), np.zeros(n)
    nc, nb = np.zeros(n, np.int32), np.zeros(n, np.int32)
    T = lights.astype(np.float64)
    e1, e2 = T[:, 1] - T[:, 0], T[:, 2] - T[:, 0]
    area2 = np.linalg.norm(np.cross(e1, e2), axis=1)
    with np.errstate(all="ignore"):
        sliver = np.where(area2 > 0, np.linalg.norm(e1, axis=1) * np.linalg.norm(e2, axis=1) / area2, np.inf)
    for i in range(n):
        rr = np.repeat(rays[i:i + 1], len(lights), 0)
        clear, border, t, w = hs.classify(lights, rr, eps, c_tol)
        dl2 = float(np.dot(rays[i, 3:].astype(np.float64), rays[i, 3:].astype(np.float64)))
        with np.errstate(all="ignore"):
            cosg = np.abs(np.einsum("i,ni->n", rays[i, 3:].astype(np.float64), np.cross(e1, e2))) / (np.sqrt(dl2) * area2)
            term = t * t * dl2 / (cosg * area2 / 2)
            tau = c_tol * u * (1 / cosg + sliver + 1) + 2 * w / np.abs(t)
        nc[i], nb[i] = clear.sum(), border.sum()
        mm = nc[i] + nb[i] + 4
        s_lo = float((term[clear] * np.maximum(0.0, 1 - tau[clear])).sum())
        hb = term[border] * (1 + tau[border])
        s_hi = float((term[clear] * (1 + tau[clear])).sum()) + (float(hb.sum()) if np.isfinite(hb).all() else np.inf)
        lo[i] = s_lo * (1 - mm * u) / len(lights)
        hi[i] = s_hi * (1 + mm * u) / len(lights)
    return lo, hi, nc, nb
