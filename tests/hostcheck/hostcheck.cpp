// hostcheck.cpp — TEST-ONLY host compilation of the device math header (csrc/pt_core.cuh) and of the
// scene re-packing (csrc/repack.h).  It lets the CPU test-suite (`-m "not gpu"`) compare the exact
// functions the CUDA kernels call (traversal, hit shading data, samplers, pdfs, BRDF, Philox lanes)
// with the oracle without a GPU.  It is NOT a render path of the product: librt_gpu.so does not
// contain or call any of this, and nothing outside tests/ builds or loads it.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "pt_core.cuh"
#include "repack.h"
#include "rt_gpu.h"

using namespace rt;

namespace {
struct HostScene {
    PackedScene p;
    DScene d;
};

bool g_rebuild = false;  // hc_set_rebuild: pack with the library's SAH builder instead of the host's tree
bool g_wide8 = false;    // hc_set_wide8: pack the 8-wide node format (its own triangle order) and trace through it

int build(const rt_scene_desc *sc, HostScene &hs) {
    if (int rc = pack_scene(*sc, hs.p, g_rebuild, g_wide8 ? RT_PACK_Q8 : RT_PACK_ALL)) return rc;
    fill_scene_constants(*sc, hs.p, hs.d);
    hs.d.scene.qnodes8 = hs.p.scene.qnodes8.data();
    hs.d.light.qnodes8 = hs.p.light.qnodes8.data();
    hs.d.scene.nodes = hs.p.scene.nodes.data();
    hs.d.scene.qnodes = hs.p.scene.qnodes.data();
    hs.d.scene.qnodes4 = hs.p.scene.qnodes4.data();
    hs.d.light.qnodes4 = hs.p.light.qnodes4.data();
    hs.d.light.qnodes = hs.p.light.qnodes.data();
    hs.d.scene.tris = hs.p.scene.tris.data();
    hs.d.light.nodes = hs.p.light.nodes.data();
    hs.d.light.tris = hs.p.light.tris.data();
    hs.d.light_sample = hs.p.light_sample.data();
    hs.d.attrs = hs.p.attrs.data();
    hs.d.tangents = hs.p.tangents.empty() ? nullptr : hs.p.tangents.data();
    hs.d.light_extra = hs.p.light_extra.data();
    hs.d.materials = hs.p.materials.data();
    hs.d.textures = hs.p.textures.data();
    hs.d.texels = hs.p.texels.data();
    return 0;
}

// the closest hit through whichever node format the scene was packed with
Hit trace(const DBvh &bvh, f3 o, f3 d, float eps) {
    return bvh.n_nodes8 ? closest_hit_q8(bvh, o, d, eps, nullptr) : closest_hit(bvh, o, d, eps);
}

Camera make_camera(const DScene &d, uint32_t w, uint32_t h) {
    Camera c;
    c.pos = mk3(d.cam_pos[0], d.cam_pos[1], d.cam_pos[2]);
    c.right = mk3(d.cam_right[0], d.cam_right[1], d.cam_right[2]);
    c.up = mk3(d.cam_up[0], d.cam_up[1], d.cam_up[2]);
    c.fwd = mk3(d.cam_fwd[0], d.cam_fwd[1], d.cam_fwd[2]);
    c.tan_half_x = tanf(d.fov_x / 2);
    const float fov_y = atanf(tanf(d.fov_x / 2) * (float)h / (float)w) * 2;
    c.tan_half_y = tanf(fov_y / 2);
    c.inv_w2 = 2.0f / (float)w;
    c.inv_h2 = 2.0f / (float)h;
    return c;
}
}  // namespace

extern "C" {

void hc_set_rebuild(int on) { g_rebuild = on != 0; }
void hc_set_wide8(int on) { g_wide8 = on != 0; }

// Worst-case k_extend stack entries of the packed 4-wide trees (out[0] scene, out[1] light); the return value is
// pack_scene's: RT_ERR_BAD_SCENE when a tree needs more than RT_EXT_STACK_CAP
int hc_stack_need(const rt_scene_desc *sc, double *out) {
    HostScene hs;
    const int rc = pack_scene(*sc, hs.p, g_rebuild, g_rebuild ? RT_PACK_Q4 : RT_PACK_ALL);
    out[0] = (double)hs.p.scene.stack_need4;
    out[1] = (double)hs.p.light.stack_need4;
    out[2] = (double)RT_EXT_STACK_CAP;
    return rc;
}

// Primary ids through the upload path's own packing: library-built tree + direct parallel 4-wide collapse
// (pack_bvh's built_tree fast path, formats = RT_PACK_Q4 only); out[0] = wide nodes, out[1] = node steps per ray
int hc_primary_ids_upload_path(const rt_scene_desc *sc, uint32_t w, uint32_t h, int32_t *ids, double *out) {
    HostScene hs;
    if (int rc = pack_scene(*sc, hs.p, true, RT_PACK_Q4)) return rc;
    fill_scene_constants(*sc, hs.p, hs.d);
    hs.d.scene.qnodes4 = hs.p.scene.qnodes4.data();
    hs.d.scene.tris = hs.p.scene.tris.data();
    const Camera cam = make_camera(hs.d, w, h);
    uint64_t steps = 0;
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            uint32_t st = 0;
            const Hit hit = closest_hit_q4(hs.d.scene, cam.pos, dir, hs.d.eps, &st);
            steps += st;
            ids[(size_t)y * w + x] = hit.tri < 0 ? -1 : (int32_t)(hs.p.scene.tris[hit.tri].id_last & ~RT_LAST_BIT);
        }
    out[0] = (double)hs.p.scene.qnodes4.size();
    out[1] = (double)steps / ((double)w * h);
    return 0;
}

// ---- containment invariant of the wide node formats ------------------------------------------------------------------
// Every decoded child box must contain every vertex (as the device forms it: a, a + e1, a + e2, evaluated exactly) of
// every triangle below that child — whatever builder, collapse and quantisation produced the tree.
namespace {
struct BoxD {
    double lo[3], hi[3];
    void reset() {
        for (int k = 0; k < 3; ++k) lo[k] = 1e300, hi[k] = -1e300;
    }
    void grow(const BoxD &b) {
        for (int k = 0; k < 3; ++k) lo[k] = std::min(lo[k], b.lo[k]), hi[k] = std::max(hi[k], b.hi[k]);
    }
};
BoxD tri_run_box(const std::vector<DTri> &tris, uint32_t first, uint32_t count_or_0, uint64_t &n_tris) {
    BoxD b;
    b.reset();
    for (uint32_t k = first;; ++k) {
        const DTri &t = tris[k];
        const double v[3][3] = {{t.ax, t.ay, t.az},
                                {(double)t.ax + t.e1x, (double)t.ay + t.e1y, (double)t.az + t.e1z},
                                {(double)t.ax + t.e2x, (double)t.ay + t.e2y, (double)t.az + t.e2z}};
        for (auto &p : v)
            for (int a = 0; a < 3; ++a) b.lo[a] = std::min(b.lo[a], p[a]), b.hi[a] = std::max(b.hi[a], p[a]);
        ++n_tris;
        if (count_or_0 ? k + 1 == first + count_or_0 : (t.id_last & RT_LAST_BIT) != 0) break;
    }
    return b;
}
double plane_of(uint32_t org_word, uint32_t byte) { return (double)u2f(org_word) + byte * ldexp(1.0, (int)(org_word & 255u) - 127); }
void check_child(const BoxD &exact, const uint32_t org[3], const uint32_t qlo[3], const uint32_t qhi[3], uint64_t &bad, uint64_t &checked) {
    for (int a = 0; a < 3; ++a) {
        ++checked;
        if (plane_of(org[a], qlo[a]) > exact.lo[a] || plane_of(org[a], qhi[a]) < exact.hi[a]) ++bad;
    }
}
BoxD walk4(const PackedBvh &b, int32_t link, uint64_t &bad, uint64_t &checked, uint64_t &n_tris, int32_t null_leaf) {
    if (link < 0) return tri_run_box(b.tris, (uint32_t)~link, 0, n_tris);
    const QNode4 &q = b.qnodes4[link];
    BoxD all;
    all.reset();
    for (int c = 0; c < 4; ++c) {
        if (q.link[c] == null_leaf) continue;
        const BoxD e = walk4(b, q.link[c], bad, checked, n_tris, null_leaf);
        const uint32_t lo[3] = {(q.lo[0] >> 8 * c) & 255u, (q.lo[1] >> 8 * c) & 255u, (q.lo[2] >> 8 * c) & 255u};
        const uint32_t hi[3] = {(q.hi[0] >> 8 * c) & 255u, (q.hi[1] >> 8 * c) & 255u, (q.hi[2] >> 8 * c) & 255u};
        check_child(e, q.org, lo, hi, bad, checked);
        all.grow(e);
    }
    return all;
}
BoxD walk8(const PackedBvh &b, uint32_t node, uint64_t &bad, uint64_t &checked, uint64_t &n_tris) {
    const QNode8 &q = b.qnodes8[node];
    BoxD all;
    all.reset();
    uint32_t rank = 0;
    for (uint32_t s = 0; s < 8; ++s) {
        const uint32_t cnt = (q.counts >> (2 * s)) & 3u;
        const bool inner = (q.imask >> s) & 1u;
        if (!inner && !cnt) continue;
        const BoxD e = inner ? walk8(b, q.child_base + rank++, bad, checked, n_tris)
                             : tri_run_box(b.tris, q.tri_base + leaf8_offset(q.counts, s), cnt, n_tris);
        const uint32_t *g = s < 4 ? q.g0 : q.g1;
        const int c = (int)(s & 3u);
        const uint32_t lo[3] = {(g[0] >> 8 * c) & 255u, (g[1] >> 8 * c) & 255u, (g[2] >> 8 * c) & 255u};
        const uint32_t hi[3] = {(g[3] >> 8 * c) & 255u, (g[4] >> 8 * c) & 255u, (g[5] >> 8 * c) & 255u};
        check_child(e, q.org, lo, hi, bad, checked);
        all.grow(e);
    }
    return all;
}
}  // namespace

// width 4 or 8; `upload_path`: pack like rt_gpu_upload_scene (library-built tree, wide format only).
// out[0] child planes checked (pairs), out[1] violations, out[2] triangles reached (must equal the scene's)
int hc_wide_containment(const rt_scene_desc *sc, int width, int upload_path, double *out) {
    PackedScene p;
    const int formats = width == 8 ? RT_PACK_Q8 : (upload_path ? RT_PACK_Q4 : RT_PACK_ALL);
    if (int rc = pack_scene(*sc, p, upload_path != 0 || g_rebuild, formats)) return rc;
    uint64_t bad = 0, checked = 0, n_tris = 0;
    for (const PackedBvh *b : {&p.scene, &p.light}) {
        if (width == 8) {
            if (!b->qnodes8.empty()) walk8(*b, 0, bad, checked, n_tris);
        } else if (b->root4 != RT_LINK_NONE) {
            walk4(*b, b->root4, bad, checked, n_tris, ~static_cast<int32_t>(b->tris.size() - 1));
        }
    }
    out[0] = (double)checked;
    out[1] = (double)bad;
    out[2] = (double)n_tris;
    return 0;
}

// Structure of the 8-wide collapse and node steps of its traversal over the pixel-centre rays:
// out[0] nodes, out[1] mean children per node, out[2] node steps per ray, out[3] triangles (must equal the scene's)
int hc_wide8_stats(const rt_scene_desc *sc, uint32_t w, uint32_t h, int32_t *ids, double *out) {
    const bool keep = g_wide8;
    g_wide8 = true;
    HostScene hs;
    const int rc = build(sc, hs);
    g_wide8 = keep;
    if (rc) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    uint64_t steps = 0;
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            uint32_t st = 0;
            const Hit hit = closest_hit_q8(hs.d.scene, cam.pos, dir, hs.d.eps, &st);
            steps += st;
            ids[(size_t)y * w + x] = hit.tri < 0 ? -1 : (int32_t)(hs.p.scene.tris[hit.tri].id_last & ~RT_LAST_BIT);
        }
    uint64_t kids = 0, tris = 0;
    for (const QNode8 &q : hs.p.scene.qnodes8) {
        kids += __builtin_popcount(q.imask & 0xFFu);
        for (int s = 0; s < 8; ++s) {
            const uint32_t c = (q.counts >> (2 * s)) & 3u;
            kids += c ? 1 : 0;
            tris += c;
        }
    }
    out[0] = (double)hs.p.scene.qnodes8.size();
    out[1] = hs.p.scene.qnodes8.empty() ? 0.0 : (double)kids / (double)hs.p.scene.qnodes8.size();
    out[2] = (double)steps / ((double)w * h);
    out[3] = (double)tris;
    return 0;
}

// Build statistics of the library's SAH builder: out[0] = seconds, out[1] = inner nodes, out[2] = leaves,
// out[3] = max leaf size, out[4] = max depth, out[5] = 1 when every triangle id appears exactly once.
// Invariants and SAH cost of a binary tree in the reference's node format over the scene's triangles (any builder:
// sah_build.h on the host, gpu_build.cuh downloaded from the device).  out[1] inner nodes, [2] leaves, [3] largest leaf,
// [4] depth, [5] 1 when every triangle sits in exactly one leaf, every leaf box is EXACTLY the union of its triangles and
// every inner box is exactly the union of its children, [6] SAH cost = (sum of inner areas + sum of leaf area x
// triangles) / root area, [7] 1 when the slots follow sah_build.h's layout (left = i + 1, right = i + 2 * n_left)
static int tree_stats(const rt_scene_desc *sc, const rt_bvh_node *nodes, size_t n_nodes, const uint32_t *objects, size_t n_objects,
                      uint32_t root, double *out) {
    double inner = 0, leaves = 0, max_leaf = 0, cost = 0;
    std::vector<int> depth(n_nodes, -1);
    std::vector<uint32_t> todo;
    int max_depth = 0;
    std::vector<uint8_t> seen(sc->n_tris, 0);
    bool once = true, layout = true;
    auto area = [](const rt_bvh_node &n) {
        const double dx = (double)n.bmax[0] - n.bmin[0], dy = (double)n.bmax[1] - n.bmin[1], dz = (double)n.bmax[2] - n.bmin[2];
        return dx * dy + dy * dz + dz * dx;
    };
    std::vector<uint32_t> count(n_nodes, 0);
    std::vector<uint32_t> order;
    if (root != RT_NO_CHILD && n_objects) {
        todo.push_back(root);
        depth[root] = 0;
    }
    while (!todo.empty()) {
        const uint32_t i = todo.back();
        todo.pop_back();
        order.push_back(i);
        const rt_bvh_node &nd = nodes[i];
        max_depth = std::max(max_depth, depth[i]);
        if (nd.left_child == RT_NO_CHILD && nd.right_child == RT_NO_CHILD) {
            ++leaves;
            if (nd.obj_end <= nd.obj_begin || nd.obj_end > n_objects) return -2;
            max_leaf = std::max(max_leaf, (double)(nd.obj_end - nd.obj_begin));
            count[i] = nd.obj_end - nd.obj_begin;
            cost += area(nd) * count[i];
            float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
            for (uint32_t k = nd.obj_begin; k < nd.obj_end; ++k) {
                const uint32_t id = objects[k];
                if (id >= sc->n_tris || seen[id]) { once = false; continue; }
                seen[id] = 1;
                for (int v = 0; v < 3; ++v)
                    for (int a = 0; a < 3; ++a) {
                        const float x = sc->tri_pos[(size_t)id * 9 + v * 3 + a];
                        lo[a] = std::min(lo[a], x);
                        hi[a] = std::max(hi[a], x);
                    }
            }
            for (int a = 0; a < 3; ++a)
                if (lo[a] != nd.bmin[a] || hi[a] != nd.bmax[a]) once = false;  // the leaf box is the union of its triangles
        } else {
            ++inner;
            cost += area(nd);
            if (nd.left_child != i + 1) layout = false;
            for (uint32_t c : {nd.left_child, nd.right_child}) {
                if (c == RT_NO_CHILD || c >= n_nodes) return -1;
                depth[c] = depth[i] + 1;
                todo.push_back(c);
            }
            const rt_bvh_node &l = nodes[nd.left_child], &r = nodes[nd.right_child];
            for (int a = 0; a < 3; ++a)
                if (std::min(l.bmin[a], r.bmin[a]) != nd.bmin[a] || std::max(l.bmax[a], r.bmax[a]) != nd.bmax[a]) once = false;
        }
    }
    for (size_t k = order.size(); k-- > 0;) {  // children were pushed after their parent: reverse order sums the counts
        const rt_bvh_node &nd = nodes[order[k]];
        if (nd.left_child != RT_NO_CHILD) {
            count[order[k]] = count[nd.left_child] + count[nd.right_child];
            if (nd.right_child != order[k] + 2 * count[nd.left_child]) layout = false;
        }
    }
    for (uint32_t id = 0; id < sc->n_tris; ++id)
        if (!seen[id] && n_objects == sc->n_tris) once = false;
    out[1] = inner; out[2] = leaves; out[3] = max_leaf; out[4] = max_depth; out[5] = once ? 1.0 : 0.0;
    out[6] = root != RT_NO_CHILD && n_objects ? cost / area(nodes[root]) : 0.0;
    out[7] = layout ? 1.0 : 0.0;
    return 0;
}

int hc_sah_stats(const rt_scene_desc *sc, double *out) {
    BuiltBvh b;
    const auto t0 = std::chrono::steady_clock::now();
    if (sc->scene_bvh.n_objects) build_sah_bvh(sc->tri_pos, sc->scene_bvh.objects, sc->scene_bvh.n_objects, b);
    else build_sah_bvh(sc->tri_pos, nullptr, sc->n_tris, b);
    out[0] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return tree_stats(sc, b.nodes.data(), b.nodes.size(), b.objects.data(), b.objects.size(), b.root, out);
}

// the same for a tree given as arrays (the device-built tree, downloaded through rt_gpu_debug_get_bvh)
int hc_tree_stats(const rt_scene_desc *sc, const rt_bvh_node *nodes, uint64_t n_nodes, const uint32_t *objects, uint64_t n_objects, double *out) {
    out[0] = 0.0;
    return tree_stats(sc, nodes, n_nodes, objects, n_objects, n_objects ? 0u : RT_NO_CHILD, out);
}

// containment invariant (walk4) of a 4-wide tree given as arrays; out as hc_wide_containment
int hc_wide_containment_arrays(const QNode4 *qnodes4, uint64_t n_nodes, int32_t root4, const DTri *tris, uint64_t n_tris_with_null, double *out) {
    PackedBvh b;
    b.qnodes4.assign(qnodes4, qnodes4 + n_nodes);
    b.tris.assign(tris, tris + n_tris_with_null);
    b.root4 = root4;
    uint64_t bad = 0, checked = 0, n_tris = 0;
    if (root4 != RT_LINK_NONE) {
        for (const QNode4 &q : b.qnodes4)
            for (int c = 0; c < 4; ++c)
                if (q.link[c] >= 0 ? (uint64_t)q.link[c] >= n_nodes : (uint64_t)(uint32_t)~q.link[c] >= n_tris_with_null) return -1;
        walk4(b, root4, bad, checked, n_tris, ~static_cast<int32_t>(b.tris.size() - 1));
    }
    out[0] = (double)checked;
    out[1] = (double)bad;
    out[2] = (double)n_tris;
    out[3] = (double)detail::stack_need4(b.qnodes4, root4, ~static_cast<int32_t>(b.tris.size() - 1));
    return 0;
}

int hc_primary_ids(const rt_scene_desc *sc, uint32_t w, uint32_t h, int32_t *ids) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            const Hit hit = trace(hs.d.scene, cam.pos, dir, hs.d.eps);
            ids[(size_t)y * w + x] = hit.tri < 0 ? -1 : (int32_t)(hs.p.scene.tris[hit.tri].id_last & ~RT_LAST_BIT);
        }
    return 0;
}

// Same through the quantised nodes in the kernel's arithmetic (closest_hit_q == what k_extend does per ray).
int hc_primary_ids_q(const rt_scene_desc *sc, uint32_t w, uint32_t h, int32_t *ids) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            const Hit hit = closest_hit_q(hs.d.scene, cam.pos, dir, hs.d.eps);
            ids[(size_t)y * w + x] = hit.tri < 0 ? -1 : (int32_t)(hs.p.scene.tris[hit.tri].id_last & ~RT_LAST_BIT);
        }
    return 0;
}

// Primary ids through the 4-wide nodes; steps[0] / steps[1] = node steps of the 4-wide / 2-wide traversal summed over
// all pixels (how many fewer, fatter steps the collapse buys).
int hc_primary_ids_q4(const rt_scene_desc *sc, uint32_t w, uint32_t h, int32_t *ids, uint64_t *steps) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    uint64_t s4 = 0, s2 = 0;
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            uint32_t st = 0;
            const Hit hit = closest_hit_q4(hs.d.scene, cam.pos, dir, hs.d.eps, &st);
            s4 += st;
            uint32_t st2 = 0;
            closest_hit_q(hs.d.scene, cam.pos, dir, hs.d.eps, &st2);
            s2 += st2;
            ids[(size_t)y * w + x] = hit.tri < 0 ? -1 : (int32_t)(hs.p.scene.tris[hit.tri].id_last & ~RT_LAST_BIT);
        }
    if (steps) {
        steps[0] = s4;
        steps[1] = s2;
    }
    return 0;
}

// Arbitrary rays (n x 6 floats: origin, direction) through the exact binary tree and through the quantised 4-wide nodes
// in the kernel's arithmetic: tri_exact / tri_q4 = the scene's triangle id or -1, t_exact / t_q4 = hit distance (inf: miss).
int hc_trace_rays(const rt_scene_desc *sc, uint64_t n, const float *rays, int32_t *tri_exact, float *t_exact, int32_t *tri_q4, float *t_q4) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    auto id = [&](int32_t k) { return k < 0 ? -1 : (int32_t)(hs.p.scene.tris[k].id_last & ~RT_LAST_BIT); };
    for (uint64_t i = 0; i < n; ++i) {
        const f3 o = mk3(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]), d = mk3(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
        const Hit a = closest_hit(hs.d.scene, o, d, hs.d.eps);
        const Hit b = closest_hit_q4(hs.d.scene, o, d, hs.d.eps, nullptr);
        tri_exact[i] = id(a.tri);
        t_exact[i] = a.t;
        tri_q4[i] = id(b.tri);
        t_q4[i] = b.t;
    }
    return 0;
}

// ---- independent closest-hit reference ----------------------------------------------------------------------------------
// Brute force over every (ray, triangle) pair in double precision, on the float32 inputs widened exactly.  It calls
// nothing from pt_core.cuh, so a defect in the shared device math cannot hide in it.  Each pair is classified against a
// LOCAL tolerance: s = c_tol * 2^-23 * (max_i |v_i - o|_inf + |t|), w = s / |cos(d, n)|.  s bounds the float32
// triangle test's rounding (relative to the magnitudes it subtracts: vertices relative to the origin, and t); dividing
// by |cos| turns it into a distance along the plane, where a grazing ray's hit point moves by error / |cos|.  s has no
// |o| term on purpose: a float32 box or triangle test whose error grows with the distance from the WORLD origin is a
// defect this reference must expose.  The tests use c_tol = 16 (tests/hit_scenarios.py); at that value the exact host
// traversal has no mismatch on any scenario.
//   clear hit:  the plane point is inside by more than w (world distance to every edge line: barycentric x altitude),
//               t > eps + w and |cos| > 1e-4;
//   clear miss: outside by more than w, or t < eps - w, or a determinant of exactly 0 (parallel ray, zero area);
//   borderline: anything else.
// Per ray: k_star = nearest clear hit (triangle index) or -1, t_star its distance, ties = clear hits with
// |t - t_star| <= w + w_star (k_star included), decidable = 1 when no borderline triangle can be closer than
// t_star + w_star (t_b - w_b < t_star + w_star) — for a ray without a clear hit: when there is no borderline pair at all.
int hc_brute_hits(const float *tri, uint64_t n_tris, const float *rays, uint64_t n_rays, double eps, double c_tol, int32_t *k_star,
                  double *t_star, int32_t *ties, uint8_t *decidable) {
    struct T {
        double v[3][3], e1[3], e2[3], n[3], area2, alt[3];
    };
    std::vector<T> tr(n_tris);
    auto len = [](const double *a) { return std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); };
    for (uint64_t k = 0; k < n_tris; ++k) {
        T &t = tr[k];
        for (int i = 0; i < 3; ++i)
            for (int a = 0; a < 3; ++a) t.v[i][a] = tri[9 * k + 3 * i + a];
        double e12[3];
        for (int a = 0; a < 3; ++a) t.e1[a] = t.v[1][a] - t.v[0][a], t.e2[a] = t.v[2][a] - t.v[0][a], e12[a] = t.v[2][a] - t.v[1][a];
        t.n[0] = t.e1[1] * t.e2[2] - t.e1[2] * t.e2[1];
        t.n[1] = t.e1[2] * t.e2[0] - t.e1[0] * t.e2[2];
        t.n[2] = t.e1[0] * t.e2[1] - t.e1[1] * t.e2[0];
        t.area2 = len(t.n);
        // altitude onto the edge opposite vertex i: the world distance of barycentric 1 from that edge
        const double l[3] = {len(e12), len(t.e2), len(t.e1)};
        for (int i = 0; i < 3; ++i) t.alt[i] = l[i] > 0 ? t.area2 / l[i] : 0.0;
    }
    auto work = [&](uint64_t r0, uint64_t r1) {
        std::vector<std::pair<double, double>> clear;  // (t, w) of the ray's clear hits
        for (uint64_t r = r0; r < r1; ++r) {
            const double o[3] = {rays[6 * r], rays[6 * r + 1], rays[6 * r + 2]}, d[3] = {rays[6 * r + 3], rays[6 * r + 4], rays[6 * r + 5]};
            const double dl = len(d);
            clear.clear();
            int32_t best = -1;
            double bt = INFINITY, bw = 0, border_lo = INFINITY;  // border_lo: min over borderline pairs of t - w
            bool any_border = false;
            for (uint64_t k = 0; k < n_tris; ++k) {
                const T &t = tr[k];
                const double det = -(d[0] * t.n[0] + d[1] * t.n[1] + d[2] * t.n[2]);
                if (det == 0.0 || t.area2 == 0.0) continue;  // clear miss
                const double y[3] = {o[0] - t.v[0][0], o[1] - t.v[0][1], o[2] - t.v[0][2]};
                const double rr[3] = {d[1] * y[2] - d[2] * y[1], d[2] * y[0] - d[0] * y[2], d[0] * y[1] - d[1] * y[0]};
                const double beta = -(t.e2[0] * rr[0] + t.e2[1] * rr[1] + t.e2[2] * rr[2]) / det;
                const double gamma = (t.e1[0] * rr[0] + t.e1[1] * rr[1] + t.e1[2] * rr[2]) / det;
                const double tt = (y[0] * t.n[0] + y[1] * t.n[1] + y[2] * t.n[2]) / det;
                double m = 0;
                for (int i = 0; i < 3; ++i)
                    for (int a = 0; a < 3; ++a) m = std::max(m, std::fabs(t.v[i][a] - o[a]));
                const double cosg = std::fabs(det) / (dl * t.area2);
                const double w = c_tol * std::ldexp(1.0, -23) * (m + std::fabs(tt)) / cosg;
                const double dist = std::min({(1.0 - beta - gamma) * t.alt[0], beta * t.alt[1], gamma * t.alt[2]});
                if (dist < -w || tt < eps - w) continue;  // clear miss
                if (dist > w && tt > eps + w && cosg > 1e-4) {
                    clear.emplace_back(tt, w);
                    if (tt < bt) bt = tt, bw = w, best = (int32_t)k;
                } else {
                    any_border = true;
                    border_lo = std::min(border_lo, tt - w);
                }
            }
            int32_t n_ties = 0;
            for (const auto &c : clear) n_ties += std::fabs(c.first - bt) <= c.second + bw ? 1 : 0;
            k_star[r] = best;
            t_star[r] = bt;
            ties[r] = n_ties;
            decidable[r] = best < 0 ? !any_border : !(border_lo < bt + bw);
        }
    };
    const unsigned n_threads = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
    std::vector<std::thread> pool;
    const uint64_t chunk = (n_rays + n_threads - 1) / n_threads;
    for (unsigned i = 0; i < n_threads; ++i) {
        const uint64_t a = std::min<uint64_t>(n_rays, i * chunk), b = std::min<uint64_t>(n_rays, a + chunk);
        if (a < b) pool.emplace_back(work, a, b);
    }
    for (auto &th : pool) th.join();
    return 0;
}

// ---- independent light-pdf reference ------------------------------------------------------------------------------------
// bvh_mix_dist::pdf of each ray by brute force over every light triangle, in double precision, sharing no code with
// pt_core.cuh.  Each (ray, light) pair is classified by hc_brute_hits' rule (clear hit / borderline / clear miss, local
// tolerance w).  A hit pair contributes term = t^2 |d|^2 / (cos * A), A = area2 / 2 of the float32 vertices, with the
// per-term relative tolerance
//   tau = c_tol * 2^-23 * (1 / cos + |e1| |e2| / |n| + 1) + 2 w / t:
// 1 / cos for the float32 cosine, |e1| |e2| / |n| for the cancellation in the cross product that gives the light's normal
// and area (the kernels' DLight record suffers it as well: slivers), 1 for the rest of the term's arithmetic, and 2 w / t
// for t^2 when t itself is only known to w.  Per ray, with m = n_clear + n_border terms:
//   lo = sum_clear term max(0, 1 - tau) (1 - (m + 4) 2^-23) / n_lights
//   hi = sum_{clear + border} term (1 + tau) (1 + (m + 4) 2^-23) / n_lights      (+inf when a borderline term is not finite)
// (m + 4) 2^-23 bounds the float32 summation of m terms, the 1 / n_lights factor and the final rounding.  A float32
// evaluation of the same sum must lie in [lo, hi]; a ray without clear and borderline pairs must give exactly 0.
int hc_brute_light_pdf(const float *tri, uint64_t n_lights, const float *rays, uint64_t n_rays, double eps, double c_tol, double *lo,
                       double *hi, int32_t *n_clear, int32_t *n_border) {
    struct T {
        double v[3][3], e1[3], e2[3], n[3], area2, alt[3], sliver;
    };
    std::vector<T> tr(n_lights);
    auto len = [](const double *a) { return std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); };
    for (uint64_t k = 0; k < n_lights; ++k) {
        T &t = tr[k];
        for (int i = 0; i < 3; ++i)
            for (int a = 0; a < 3; ++a) t.v[i][a] = tri[9 * k + 3 * i + a];
        double e12[3];
        for (int a = 0; a < 3; ++a) t.e1[a] = t.v[1][a] - t.v[0][a], t.e2[a] = t.v[2][a] - t.v[0][a], e12[a] = t.v[2][a] - t.v[1][a];
        t.n[0] = t.e1[1] * t.e2[2] - t.e1[2] * t.e2[1];
        t.n[1] = t.e1[2] * t.e2[0] - t.e1[0] * t.e2[2];
        t.n[2] = t.e1[0] * t.e2[1] - t.e1[1] * t.e2[0];
        t.area2 = len(t.n);
        const double l[3] = {len(e12), len(t.e2), len(t.e1)};
        for (int i = 0; i < 3; ++i) t.alt[i] = l[i] > 0 ? t.area2 / l[i] : 0.0;
        t.sliver = t.area2 > 0 ? l[1] * l[2] / t.area2 : INFINITY;
    }
    const double u = std::ldexp(1.0, -23);
    const double inv_n = n_lights ? 1.0 / (double)n_lights : 0.0;
    auto work = [&](uint64_t r0, uint64_t r1) {
        for (uint64_t r = r0; r < r1; ++r) {
            const double o[3] = {rays[6 * r], rays[6 * r + 1], rays[6 * r + 2]}, d[3] = {rays[6 * r + 3], rays[6 * r + 4], rays[6 * r + 5]};
            const double dl = len(d);
            double s_lo = 0, s_hi = 0;
            int32_t nc = 0, nb = 0;
            for (uint64_t k = 0; k < n_lights; ++k) {
                const T &t = tr[k];
                const double det = -(d[0] * t.n[0] + d[1] * t.n[1] + d[2] * t.n[2]);
                if (det == 0.0 || t.area2 == 0.0) continue;  // clear miss
                const double y[3] = {o[0] - t.v[0][0], o[1] - t.v[0][1], o[2] - t.v[0][2]};
                const double rr[3] = {d[1] * y[2] - d[2] * y[1], d[2] * y[0] - d[0] * y[2], d[0] * y[1] - d[1] * y[0]};
                const double beta = -(t.e2[0] * rr[0] + t.e2[1] * rr[1] + t.e2[2] * rr[2]) / det;
                const double gamma = (t.e1[0] * rr[0] + t.e1[1] * rr[1] + t.e1[2] * rr[2]) / det;
                const double tt = (y[0] * t.n[0] + y[1] * t.n[1] + y[2] * t.n[2]) / det;
                double m = 0;
                for (int i = 0; i < 3; ++i)
                    for (int a = 0; a < 3; ++a) m = std::max(m, std::fabs(t.v[i][a] - o[a]));
                const double cosg = std::fabs(det) / (dl * t.area2);
                const double w = c_tol * u * (m + std::fabs(tt)) / cosg;
                const double dist = std::min({(1.0 - beta - gamma) * t.alt[0], beta * t.alt[1], gamma * t.alt[2]});
                if (dist < -w || tt < eps - w) continue;  // clear miss
                const double term = tt * tt * dl * dl / (cosg * t.area2 / 2);
                const double tau = c_tol * u * (1 / cosg + t.sliver + 1) + 2 * w / std::fabs(tt);
                if (dist > w && tt > eps + w && cosg > 1e-4) {
                    ++nc;
                    s_lo += term * std::max(0.0, 1 - tau);
                    s_hi += term * (1 + tau);
                } else {
                    ++nb;
                    s_hi += std::isfinite(term) && std::isfinite(tau) ? term * (1 + tau) : INFINITY;
                }
            }
            const double mm = (double)(nc + nb) + 4;
            lo[r] = s_lo * (1 - mm * u) * inv_n;
            hi[r] = s_hi * (1 + mm * u) * inv_n;
            n_clear[r] = nc;
            n_border[r] = nb;
        }
    };
    const unsigned n_threads = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
    std::vector<std::thread> pool;
    const uint64_t chunk = (n_rays + n_threads - 1) / n_threads;
    for (unsigned i = 0; i < n_threads; ++i) {
        const uint64_t a = std::min<uint64_t>(n_rays, i * chunk), b = std::min<uint64_t>(n_rays, a + chunk);
        if (a < b) pool.emplace_back(work, a, b);
    }
    for (auto &th : pool) th.join();
    return 0;
}

// The light pdf (bvh_mix_dist::pdf, 1 / n_lights included) of arbitrary rays (n x 6 floats: origin, direction) through the
// host compilation of the device math, the scene packed as hc_render packs it: pdf_exact = light_pdf over the exact
// binary light nodes, pdf_q8 = light_pdf_q8 over the 8-wide quantised light nodes.  A scene without lights gives 0.
int hc_light_pdf(const rt_scene_desc *sc, uint64_t n, const float *rays, float *pdf_exact, float *pdf_q8) {
    const bool keep = g_wide8;
    for (int pass = 0; pass < 2; ++pass) {
        HostScene hs;
        g_wide8 = pass == 1;
        const int rc = build(sc, hs);
        g_wide8 = keep;
        if (rc) return rc;
        if ((pass == 1) != (hs.d.light.n_nodes8 != 0) && hs.d.n_lights) return -100;  // not the node format asked for
        float *out = pass ? pdf_q8 : pdf_exact;
        for (uint64_t i = 0; i < n; ++i) {
            const f3 o = mk3(rays[6 * i], rays[6 * i + 1], rays[6 * i + 2]), d = mk3(rays[6 * i + 3], rays[6 * i + 4], rays[6 * i + 5]);
            out[i] = hs.d.n_lights ? light_pdf(hs.d, o, d) : 0.0f;
        }
    }
    return 0;
}

// Wall time of the re-pack phases (ms): out[0] SAH build, out[1] pack_bvh of the scene tree (triangles, nodes, both
// quantisations, collapse), out[2] whole pack_scene with rebuild, out[3] the upload path's pack_scene (4-wide only),
// out[4..7] its phases.
int hc_pack_timing(const rt_scene_desc *sc, double *out) {
    using clk = std::chrono::steady_clock;
    auto ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    auto t0 = clk::now();
    BuiltBvh built;
    build_sah_bvh(sc->tri_pos, sc->scene_bvh.objects, sc->scene_bvh.n_objects, built);
    auto t1 = clk::now();
    PackedBvh pb;
    if (int rc = pack_bvh(*sc, built.desc(), pb)) return rc;
    auto t2 = clk::now();
    PackedScene ps;
    if (int rc = pack_scene(*sc, ps, true)) return rc;
    auto t3 = clk::now();
    PackedScene pq;
    double phase[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    pack_times() = phase;
    const int rq = pack_scene(*sc, pq, true, RT_PACK_Q4);  // what rt_gpu_upload_scene runs
    pack_times() = nullptr;
    if (rq) return rq;
    auto t4 = clk::now();
    out[0] = ms(t0, t1); out[1] = ms(t1, t2); out[2] = ms(t2, t3); out[3] = ms(t3, t4);
    for (int k = 0; k < 4; ++k) out[4 + k] = phase[k];  // SAH build, triangles (+ binary nodes), collapse, quantise
    return 0;
}

// Quantised-node invariants over the whole scene BVH.  out[0] = nodes, out[1] = planes whose decoded position
// (exact arithmetic: org + q * cell) is on the wrong side of the exact plane (must be 0), out[2] = planes with
// less than 1/128 cell of slack (must be 0: the packer keeps 1/64), out[3..4] = summed surface area of the exact
// / decoded child boxes (how much looser the quantised tree is).
int hc_qnode_check(const rt_scene_desc *sc, double *out) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const PackedBvh &b = hs.p.scene;
    if (b.qnodes.size() != b.nodes.size()) return -100;
    double bad = 0, tight = 0, area_exact = 0, area_q = 0;
    for (size_t i = 0; i < b.nodes.size(); ++i) {
        const DNode &n = b.nodes[i];
        const QNode &q = b.qnodes[i];
        if (q.left != n.left || q.right != n.right) return -101;
        const float exact[12] = {n.lminx, n.lminy, n.lminz, n.lmaxx, n.lmaxy, n.lmaxz,
                                 n.rminx, n.rminy, n.rminz, n.rmaxx, n.rmaxy, n.rmaxz};
        double dec[12];
        for (int k = 0; k < 12; ++k) {  // k = DNode plane order: child (k / 6), min/max ((k / 3) & 1), axis (k % 3)
            const int axis = k % 3;
            const bool is_max = (k / 3) & 1;
            const int child = k / 6;
            const uint32_t word = q.org[axis];
            if (word & 0x100u) return -102;
            const double org = (double)u2f(word), cell = ldexp(1.0, (int)(word & 255u) - 127);
            const uint32_t byte = (q.q[axis] >> (8 * (2 * child + (is_max ? 1 : 0)))) & 255u;
            dec[k] = org + byte * cell;
            const double slack = is_max ? dec[k] - (double)exact[k] : (double)exact[k] - dec[k];
            if (slack < 0) ++bad;
            else if (slack < cell / 128) ++tight;
        }
        for (int c = 0; c < 2; ++c) {
            const float *e = exact + 6 * c;
            const double *d = dec + 6 * c;
            const double ex = e[3] - e[0], ey = e[4] - e[1], ez = e[5] - e[2];
            const double dx = d[3] - d[0], dy = d[4] - d[1], dz = d[5] - d[2];
            area_exact += 2 * (ex * ey + ey * ez + ez * ex);
            area_q += 2 * (dx * dy + dy * dz + dz * dx);
        }
    }
    out[0] = (double)b.nodes.size();
    out[1] = bad;
    out[2] = tight;
    out[3] = area_exact;
    out[4] = area_q;
    return 0;
}

// Surface of the primary hit per pixel, 18 floats in the layout of `ref_tool hitinfo`.
int hc_hitinfo(const rt_scene_desc *sc, uint32_t w, uint32_t h, float *out) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    std::memset(out, 0, (size_t)w * h * 18 * sizeof(float));
    for (uint32_t y = 0; y < h; ++y)
        for (uint32_t x = 0; x < w; ++x) {
            const f3 dir = camera_dir(cam, (float)x + 0.5f, (float)y + 0.5f);
            const Hit hit = trace(hs.d.scene, cam.pos, dir, hs.d.eps);
            if (hit.tri < 0) continue;
            const Surface sf = make_surface(hs.d, hs.p.gamma_lut, hit, dir);
            float *o = out + ((size_t)y * w + x) * 18;
            o[0] = hit.t;
            o[1] = sf.ng.x; o[2] = sf.ng.y; o[3] = sf.ng.z;
            o[4] = sf.ns.x; o[5] = sf.ns.y; o[6] = sf.ns.z;
            o[7] = sf.color.x; o[8] = sf.color.y; o[9] = sf.color.z; o[10] = sf.alpha;
            o[11] = sf.emission.x; o[12] = sf.emission.y; o[13] = sf.emission.z;
            o[14] = sf.metallic; o[15] = sf.roughness;
            o[16] = 0.0f;  // is_inside is folded into the normals
            o[17] = sf.ior;
        }
    return 0;
}

// Sequential per-sample loop over the same state transition the wavefront kernels apply.
int hc_render(const rt_scene_desc *sc, uint32_t w, uint32_t h, uint32_t samples, uint32_t s_begin, uint32_t s_end,
              uint64_t seed, float *rgb_mean, uint64_t *counters /* ext rays, light rays */) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    uint64_t ext = 0, lrays = 0;
    for (uint32_t pix = 0; pix < w * h; ++pix) {
        f3 sum = mk3(0, 0, 0);
        for (uint32_t s = s_begin; s < s_end; ++s) {
            const RngKey key{pix, s, (uint32_t)seed, (uint32_t)(seed >> 32)};
            const u4 j = rng_jitter(key);
            f3 o = cam.pos;
            f3 d = camera_dir(cam, (float)(pix % w) + u01(j.x), (float)(pix / w) + u01(j.y));
            f3 thr = mk3(1, 1, 1), rad = mk3(0, 0, 0);
            for (uint32_t b = 0; b < hs.d.ray_depth; ++b) {
                const Hit hit = trace(hs.d.scene, o, d, hs.d.eps);
                ++ext;
                uint32_t lr = 0;
                const bool alive = shade_bounce(hs.d, hs.p.gamma_lut, key, b, b + 1 == hs.d.ray_depth, hit, o, d, thr, rad, lr);
                lrays += lr;
                if (!alive) break;
            }
            sum = sum + sanitize(rad);
        }
        rgb_mean[(size_t)pix * 3 + 0] = sum.x / (float)samples;
        rgb_mean[(size_t)pix * 3 + 1] = sum.y / (float)samples;
        rgb_mean[(size_t)pix * 3 + 2] = sum.z / (float)samples;
    }
    if (counters) {
        counters[0] = ext;
        counters[1] = lrays;
    }
    return 0;
}

void hc_philox(const uint32_t *ctr, const uint32_t *key, uint32_t *out) {
    const u4 r = philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

}  // extern "C"
