// repack.h — host-side re-packing of an rt_scene_desc (reference layout) into the device layout of
// rt_types.h.  Pure C++ (no CUDA), header-only; used by rt_gpu_upload_scene and by the host unit
// test of the device math (tests/hostcheck).
#ifndef RT_REPACK_H
#define RT_REPACK_H

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <limits>
#include <thread>
#include <vector>

#include "quantize.h"
#include "rt_gpu.h"
#include "rt_types.h"
#include "sah_build.h"

namespace rt {

struct PackedBvh {
    std::vector<DNode> nodes;
    std::vector<QNode> qnodes;    // quantised copy of `nodes` (same indices), see quantize_nodes()
    std::vector<QNode4> qnodes4;  // 4-wide collapse of the same tree (own indices), see collapse4()
    int32_t root4 = RT_LINK_NONE;
    std::vector<QNode8> qnodes8;  // 8-wide collapse (RT_PACK_Q8 only: `tris` / `order` are then in ITS triangle order and
                                  // the 2- and 4-wide arrays are not produced); node 0 is the root
    std::vector<DTri> tris;       // BVH object order
    std::vector<uint32_t> order;  // BVH position -> scene.objects index
    int32_t root = RT_LINK_NONE;
    uint32_t max_depth = 0;
    uint32_t stack_need4 = 0;     // worst-case traversal-stack entries of a ray through qnodes4 (stack_need4())
};

struct PackedScene {
    PackedBvh scene, light;
    std::vector<DAttr> attrs;
    std::vector<DTangent> tangents;  // empty when every tangent is (1,0,0)
    std::vector<DLight> light_extra;
    std::vector<DTri> light_sample;  // emissive triangles in the host light BVH's object order (sampling order)
    std::vector<DMat> materials;
    std::vector<DTex> textures;
    std::vector<uint32_t> texels;
    float gamma_lut[256];  // powf(k/255, 2.2f): the per-texel pow of Texture::sample (geometry.h:525-527,561)
    // working memory of the library's BVH builder, kept with the staging arrays (re-used by the next pack_scene)
    BuiltBvh built;
    sah::Ctx sah_scratch;
};

// optional phase timers (ms) of pack_scene, for RT_TIMING=1 and the host timing test: [0] SAH build (scene),
// [1] triangles + binary nodes, [2] wide collapse, [3] quantisation, [4] light BVHs, [5] attributes, [6] materials/texels
inline double *&pack_times() {
    static thread_local double *p = nullptr;
    return p;
}
struct PackLap {
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(int slot) {
        const auto n = std::chrono::steady_clock::now();
        if (pack_times()) pack_times()[slot] += std::chrono::duration<double, std::milli>(n - t).count();
        t = n;
    }
};

namespace detail {

// run fn(begin, end) over [0, n) on up to `max_threads` host threads (the per-node packing loops are independent)
template <class F> inline void parallel_for(size_t n, F fn, size_t grain = 4096, unsigned max_threads = 16) {
    unsigned hw = std::thread::hardware_concurrency();
    size_t nt = std::min<size_t>(std::min<unsigned>(hw ? hw : 1, max_threads), (n + grain - 1) / grain);
    if (nt <= 1) {
        fn(static_cast<size_t>(0), n);
        return;
    }
    std::vector<std::thread> th;
    const size_t chunk = (n + nt - 1) / nt;
    for (size_t t = 1; t < nt; ++t) th.emplace_back([=] { fn(std::min(n, t * chunk), std::min(n, (t + 1) * chunk)); });
    fn(static_cast<size_t>(0), std::min(n, chunk));
    for (auto &x : th) x.join();
}

inline void set_box(DNode &n, bool left, const float *lo, const float *hi) {
    if (left) {
        n.lminx = lo[0]; n.lminy = lo[1]; n.lminz = lo[2];
        n.lmaxx = hi[0]; n.lmaxy = hi[1]; n.lmaxz = hi[2];
    } else {
        n.rminx = lo[0]; n.rminy = lo[1]; n.rminz = lo[2];
        n.rmaxx = hi[0]; n.rmaxy = hi[1]; n.rmaxz = hi[2];
    }
}

inline bool subtree_empty(const rt_bvh_desc &src, uint32_t ref_id, uint32_t depth) {
    if (ref_id == RT_NO_CHILD) return true;
    if (depth > RT_STACK_SIZE) return false;  // malformed (cyclic) input: reported by pack_node's depth check
    const rt_bvh_node &nd = src.nodes[ref_id];
    if (nd.left_child == RT_NO_CHILD && nd.right_child == RT_NO_CHILD) return nd.obj_begin >= nd.obj_end;
    return subtree_empty(src, nd.left_child, depth + 1) && subtree_empty(src, nd.right_child, depth + 1);
}

// Returns the link of reference node `ref_id` (inner index or ~first_tri), or RT_LINK_NONE for an
// empty subtree.  An inner node with one empty side (the reference builder never makes one) is replaced
// by its other child, so every packed inner node has two non-empty children.  `rc` collects structural errors.
inline int32_t pack_node(const rt_bvh_desc &src, uint32_t ref_id, PackedBvh &out, uint32_t depth, int &rc) {
    const rt_bvh_node &nd = src.nodes[ref_id];
    if (depth > out.max_depth) out.max_depth = depth;
    const bool has_children = nd.left_child != RT_NO_CHILD || nd.right_child != RT_NO_CHILD;
    if (has_children && depth < RT_STACK_SIZE && nd.obj_begin >= nd.obj_end) {
        const bool el = subtree_empty(src, nd.left_child, depth + 1), er = subtree_empty(src, nd.right_child, depth + 1);
        if (el && er) return RT_LINK_NONE;
        if (el || er) return pack_node(src, el ? nd.right_child : nd.left_child, out, depth + 1, rc);
    }
    if (!has_children) {
        if (nd.obj_begin >= nd.obj_end) return RT_LINK_NONE;
        out.tris[nd.obj_end - 1].id_last |= RT_LAST_BIT;
        return ~static_cast<int32_t>(nd.obj_begin);
    }
    if (nd.obj_begin < nd.obj_end || depth >= RT_STACK_SIZE) {
        rc = RT_ERR_BAD_SCENE;  // inner node with own objects / deeper than bvh.h:371 allows
        return RT_LINK_NONE;
    }
    const int32_t idx = static_cast<int32_t>(out.nodes.size());
    out.nodes.emplace_back();
    const float inf = std::numeric_limits<float>::infinity();
    const float empty_lo[3] = {inf, inf, inf}, empty_hi[3] = {-inf, -inf, -inf};
    int32_t links[2];
    const uint32_t child[2] = {nd.left_child, nd.right_child};
    for (int c = 0; c < 2; ++c) {
        if (child[c] == RT_NO_CHILD) {
            links[c] = RT_LINK_NONE;
            set_box(out.nodes[idx], c == 0, empty_lo, empty_hi);
        } else {
            links[c] = pack_node(src, child[c], out, depth + 1, rc);
            const rt_bvh_node &ch = src.nodes[child[c]];
            if (links[c] == RT_LINK_NONE)
                set_box(out.nodes[idx], c == 0, empty_lo, empty_hi);
            else
                set_box(out.nodes[idx], c == 0, ch.bmin, ch.bmax);
        }
    }
    out.nodes[idx].left = links[0];
    out.nodes[idx].right = links[1];
    out.nodes[idx].pad0 = out.nodes[idx].pad1 = 0;
    return idx;
}

inline bool quantize_axis(const float lo[2], const float hi[2], uint32_t &word, uint8_t q[4]) {
    uint8_t ql[2], qh[2];
    if (!quantize_axis_n(lo, hi, 2, word, ql, qh)) return false;
    q[0] = ql[0]; q[1] = qh[0]; q[2] = ql[1]; q[3] = qh[1];
    return true;
}

inline int quantize_nodes(const std::vector<DNode> &nodes, std::vector<QNode> &out) {
    out.resize(nodes.size());
    std::atomic<int> rc{RT_OK};
    parallel_for(nodes.size(), [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const DNode &n = nodes[i];
            const float lo[3][2] = {{n.lminx, n.rminx}, {n.lminy, n.rminy}, {n.lminz, n.rminz}};
            const float hi[3][2] = {{n.lmaxx, n.rmaxx}, {n.lmaxy, n.rmaxy}, {n.lmaxz, n.rmaxz}};
            uint8_t q[3][4];
            QNode &o = out[i];
            for (int a = 0; a < 3; ++a)
                if (!quantize_axis(lo[a], hi[a], o.org[a], q[a])) rc = RT_ERR_BAD_SCENE;
            // one word per axis: left.min, left.max, right.min, right.max (quantize_axis's order)
            for (int w = 0; w < 3; ++w)
                o.q[w] = static_cast<uint32_t>(q[w][0]) | static_cast<uint32_t>(q[w][1]) << 8 |
                         static_cast<uint32_t>(q[w][2]) << 16 | static_cast<uint32_t>(q[w][3]) << 24;
            o.left = n.left;
            o.right = n.right;
        }
    });
    return rc;
}

// ---- 4-wide collapse ------------------------------------------------------------------------------------------
struct Child4 {
    int32_t link;
    float lo[3], hi[3];
};
inline float box_area(const Child4 &c) {
    const float dx = c.hi[0] - c.lo[0], dy = c.hi[1] - c.lo[1], dz = c.hi[2] - c.lo[2];
    return dx * dy + dy * dz + dz * dx;
}
inline void children_of(const DNode &n, Child4 out[2]) {
    out[0] = Child4{n.left, {n.lminx, n.lminy, n.lminz}, {n.lmaxx, n.lmaxy, n.lmaxz}};
    out[1] = Child4{n.right, {n.rminx, n.rminy, n.rminz}, {n.rmaxx, n.rmaxy, n.rmaxz}};
}
// Returns the 4-wide link of binary link `link` (leaves keep their ~first_triangle link).  Only the topology is built
// here (children and their exact boxes, recorded in `boxes`); quantise_nodes4() fills the plane bytes afterwards.
struct Node4Boxes {
    Child4 ch[4];
    int n;
};
inline int32_t collapse4(const std::vector<DNode> &nodes, int32_t link, int32_t null_leaf, std::vector<QNode4> &out,
                         std::vector<Node4Boxes> &boxes) {
    if (link < 0) return link;
    Node4Boxes nb;
    nb.n = 2;
    children_of(nodes[link], nb.ch);
    while (nb.n < 4) {  // open the inner child with the largest box until four children or only leaves are left
        int best = -1;
        float best_area = -1.0f;
        for (int i = 0; i < nb.n; ++i)
            if (nb.ch[i].link >= 0 && box_area(nb.ch[i]) > best_area) {
                best_area = box_area(nb.ch[i]);
                best = i;
            }
        if (best < 0) break;
        Child4 two[2];
        children_of(nodes[nb.ch[best].link], two);
        nb.ch[best] = two[0];
        nb.ch[nb.n++] = two[1];
    }
    const int32_t idx = static_cast<int32_t>(out.size());
    out.emplace_back();
    boxes.push_back(nb);
    int32_t links[4];
    for (int i = 0; i < 4; ++i) links[i] = i < nb.n ? collapse4(nodes, nb.ch[i].link, null_leaf, out, boxes) : null_leaf;
    QNode4 &q = out[idx];
    std::memset(&q, 0, sizeof q);
    for (int i = 0; i < 4; ++i) q.link[i] = links[i];
    return idx;
}
inline int quantize_nodes4(const std::vector<Node4Boxes> &boxes, std::vector<QNode4> &out) {
    std::atomic<int> rc{RT_OK};
    parallel_for(out.size(), [&](size_t b, size_t e) {
        for (size_t k = b; k < e; ++k) {
            const Node4Boxes &nb = boxes[k];
            QNode4 &q = out[k];
            for (int a = 0; a < 3; ++a) {
                float lo[4], hi[4];
                uint8_t ql[4] = {255, 255, 255, 255}, qh[4] = {0, 0, 0, 0};  // absent child: inverted box
                for (int i = 0; i < nb.n; ++i) {
                    lo[i] = nb.ch[i].lo[a];
                    hi[i] = nb.ch[i].hi[a];
                }
                if (!quantize_axis_n(lo, hi, nb.n, q.org[a], ql, qh)) rc = RT_ERR_BAD_SCENE;
                q.lo[a] = static_cast<uint32_t>(ql[0]) | static_cast<uint32_t>(ql[1]) << 8 | static_cast<uint32_t>(ql[2]) << 16 |
                          static_cast<uint32_t>(ql[3]) << 24;
                q.hi[a] = static_cast<uint32_t>(qh[0]) | static_cast<uint32_t>(qh[1]) << 8 | static_cast<uint32_t>(qh[2]) << 16 |
                          static_cast<uint32_t>(qh[3]) << 24;
            }
        }
    });
    return rc;
}

// Worst-case number of traversal-stack entries a ray can hold in the 4-wide tree: a node step pushes every hit child but
// the nearest (at most children - 1) and descends, so the need below a node is the sum of (children - 1) over its
// ancestors and itself.  Both collapses number a child after its parent, so one forward pass does it.  k_extend's stack
// holds RT_EXT_STACK_CAP entries and does not check: pack_bvh rejects a deeper tree (a degenerate chain from a host
// builder with overlapping boxes can reach 3 entries per binary level).
inline uint32_t stack_need4(const std::vector<QNode4> &nodes, int32_t root4, int32_t null_leaf) {
    if (root4 < 0 || root4 == RT_LINK_NONE || nodes.empty()) return 0;
    std::vector<uint32_t> above(nodes.size(), 0);
    uint32_t worst = 0;
    for (size_t i = 0; i < nodes.size(); ++i) {
        const QNode4 &q = nodes[i];
        uint32_t n_real = 0;
        for (int c = 0; c < 4; ++c) n_real += q.link[c] != null_leaf ? 1u : 0u;
        const uint32_t below = above[i] + (n_real ? n_real - 1 : 0);
        worst = std::max(worst, below);
        for (int c = 0; c < 4; ++c)
            if (q.link[c] >= 0 && static_cast<size_t>(q.link[c]) > i) above[q.link[c]] = below;
    }
    return worst;
}

// ---- 4-wide collapse straight from a tree of the library's own builder, sub-trees in parallel ------------------------
// sah_build.h's trees are well formed (every inner node has two non-empty children, a leaf holds [obj_begin, obj_end)),
// so the binary DNode array and its serial construction (pack_node) are skipped on the upload path: the wide nodes of
// the top three levels are made serially, the sub-trees below them by one task each into private arrays that are
// appended afterwards (inner links shifted by the task's base index).
struct Built4 {
    const rt_bvh_desc &src;
    std::vector<DTri> &tris;
    int32_t null_leaf;
    // link of binary node i for the collapse: >= 0 = i itself (inner), < 0 = ~first triangle (leaf; its last triangle is marked)
    int32_t link_of(uint32_t i) const {
        const rt_bvh_node &nd = src.nodes[i];
        if (nd.left_child == RT_NO_CHILD && nd.right_child == RT_NO_CHILD) {
            tris[nd.obj_end - 1].id_last |= RT_LAST_BIT;
            return ~static_cast<int32_t>(nd.obj_begin);
        }
        return static_cast<int32_t>(i);
    }
    Child4 child(uint32_t i) const {
        const rt_bvh_node &nd = src.nodes[i];
        return Child4{link_of(i), {nd.bmin[0], nd.bmin[1], nd.bmin[2]}, {nd.bmax[0], nd.bmax[1], nd.bmax[2]}};
    }
    // the 2..4 children of the wide node rooted at binary inner node `bin` (largest box opened first, as collapse4)
    Node4Boxes open(int32_t bin) const {
        Node4Boxes nb;
        nb.n = 2;
        nb.ch[0] = child(src.nodes[bin].left_child);
        nb.ch[1] = child(src.nodes[bin].right_child);
        while (nb.n < 4) {
            int best = -1;
            float best_area = -1.0f;
            for (int i = 0; i < nb.n; ++i)
                if (nb.ch[i].link >= 0 && box_area(nb.ch[i]) > best_area) {
                    best_area = box_area(nb.ch[i]);
                    best = i;
                }
            if (best < 0) break;
            const rt_bvh_node &nd = src.nodes[nb.ch[best].link];
            nb.ch[best] = child(nd.left_child);
            nb.ch[nb.n++] = child(nd.right_child);
        }
        return nb;
    }
    // serial collapse of a sub-tree into (out, boxes); returns its root's index in `out`
    int32_t collapse(int32_t bin, std::vector<QNode4> &out, std::vector<Node4Boxes> &boxes) const {
        const Node4Boxes nb = open(bin);
        const int32_t idx = static_cast<int32_t>(out.size());
        out.emplace_back();
        boxes.push_back(nb);
        int32_t links[4];
        for (int i = 0; i < 4; ++i)
            links[i] = i < nb.n ? (nb.ch[i].link >= 0 ? collapse(nb.ch[i].link, out, boxes) : nb.ch[i].link) : null_leaf;
        QNode4 &q = out[idx];
        std::memset(&q, 0, sizeof q);
        for (int i = 0; i < 4; ++i) q.link[i] = links[i];
        return idx;
    }
};
inline int32_t collapse4_built(const rt_bvh_desc &src, std::vector<DTri> &tris, int32_t null_leaf, std::vector<QNode4> &out,
                               std::vector<Node4Boxes> &boxes) {
    const Built4 b{src, tris, null_leaf};
    const int32_t root_link = b.link_of(src.root);
    if (root_link < 0) return root_link;  // the whole tree is one leaf
    struct Task {
        int32_t bin;
        uint32_t parent;
        int slot;
        std::vector<QNode4> nodes;
        std::vector<Node4Boxes> boxes;
    };
    std::vector<Task> tasks;
    // top levels, breadth first: (binary node, wide parent, slot, depth)
    struct Top {
        int32_t bin;
        uint32_t parent;
        int slot, depth;
    };
    std::vector<Top> queue{{root_link, 0u, -1, 0}};
    for (size_t qi = 0; qi < queue.size(); ++qi) {
        const Top t = queue[qi];
        const Node4Boxes nb = b.open(t.bin);
        const uint32_t idx = static_cast<uint32_t>(out.size());
        out.emplace_back();
        boxes.push_back(nb);
        std::memset(&out[idx], 0, sizeof(QNode4));
        if (t.slot >= 0) out[t.parent].link[t.slot] = static_cast<int32_t>(idx);
        for (int i = 0; i < 4; ++i) {
            if (i >= nb.n) {
                out[idx].link[i] = null_leaf;
            } else if (nb.ch[i].link < 0) {
                out[idx].link[i] = nb.ch[i].link;
            } else if (t.depth < 2) {
                queue.push_back({nb.ch[i].link, idx, i, t.depth + 1});
            } else {
                tasks.emplace_back();
                tasks.back().bin = nb.ch[i].link;
                tasks.back().parent = idx;
                tasks.back().slot = i;
            }
        }
    }
    // sub-trees in parallel (dynamic hand-out: their sizes differ)
    std::atomic<size_t> next{0};
    const unsigned hw = std::thread::hardware_concurrency();
    const size_t nt = std::min<size_t>(std::min<unsigned>(hw ? hw : 1, 16), tasks.size());
    auto worker = [&] {
        for (size_t k = next++; k < tasks.size(); k = next++) b.collapse(tasks[k].bin, tasks[k].nodes, tasks[k].boxes);
    };
    std::vector<std::thread> th;
    for (size_t t = 1; t < nt; ++t) th.emplace_back(worker);
    worker();
    for (auto &x : th) x.join();
    // append: task k's nodes start at base[k]
    std::vector<size_t> base(tasks.size() + 1, out.size());
    for (size_t k = 0; k < tasks.size(); ++k) base[k + 1] = base[k] + tasks[k].nodes.size();
    out.resize(base.back());
    boxes.resize(base.back());
    next = 0;
    auto copier = [&] {
        for (size_t k = next++; k < tasks.size(); k = next++) {
            const int32_t off = static_cast<int32_t>(base[k]);
            for (size_t i = 0; i < tasks[k].nodes.size(); ++i) {
                QNode4 q = tasks[k].nodes[i];
                for (int c = 0; c < 4; ++c)
                    if (q.link[c] >= 0) q.link[c] += off;
                out[base[k] + i] = q;
                boxes[base[k] + i] = tasks[k].boxes[i];
            }
            out[tasks[k].parent].link[tasks[k].slot] = off;  // the sub-tree's root is its first node
        }
    };
    th.clear();
    for (size_t t = 1; t < nt; ++t) th.emplace_back(copier);
    copier();
    for (auto &x : th) x.join();
    return 0;
}

// ---- 8-wide collapse (QNode8) ---------------------------------------------------------------------------------
constexpr uint32_t kLeaf8 = 3;  // triangles per leaf child (2 count bits per slot)
#ifndef RT_COLLAPSE8_OPTIMAL
#define RT_COLLAPSE8_OPTIMAL 1  // 1: cost-optimal collapse (6.0 of 8 slots filled on the bench scene)  0: greedy (4.5)
#endif
struct Item8 {
    int32_t link;     // >= 0: inner node of the binary tree; < 0: the triangle range [tb, te) (BVH-order positions)
    uint32_t tb, te;
    float lo[3], hi[3];
    bool openable() const { return link >= 0 || te - tb > kLeaf8; }
};
struct Node8Boxes {
    float lo[8][3], hi[8][3];
    uint8_t present;
};
inline float box_area(const Item8 &c) {
    const float dx = c.hi[0] - c.lo[0], dy = c.hi[1] - c.lo[1], dz = c.hi[2] - c.lo[2];
    return dx * dy + dy * dz + dz * dx;
}
struct Collapse8 {
    const std::vector<DNode> &nodes;
    const std::vector<DTri> &tris;  // BVH order, RT_LAST_BIT marks the ends of the binary leaves
    std::vector<QNode8> &out;
    std::vector<Node8Boxes> &boxes;
    std::vector<uint32_t> &perm;  // new triangle position -> old (BVH-order) position
    std::vector<uint32_t> &last;  // new positions that end a leaf child

    Item8 range_item(uint32_t tb, uint32_t te) const {
        Item8 it;
        it.link = -1;
        it.tb = tb;
        it.te = te;
        const float inf = std::numeric_limits<float>::infinity();
        for (int k = 0; k < 3; ++k) it.lo[k] = inf, it.hi[k] = -inf;
        for (uint32_t i = tb; i < te; ++i) {
            const DTri &t = tris[i];
            const float a[3] = {t.ax, t.ay, t.az}, e1[3] = {t.e1x, t.e1y, t.e1z}, e2[3] = {t.e2x, t.e2y, t.e2z};
            for (int k = 0; k < 3; ++k) {
                // the vertices as the builders saw them: b = a + (b - a) may differ from b in the last bit, so the box
                // takes both roundings into account by a one-ulp widening
                const float v1 = a[k] + e1[k], v2 = a[k] + e2[k];
                const float mn = std::min(a[k], std::min(v1, v2)), mx = std::max(a[k], std::max(v1, v2));
                it.lo[k] = std::min(it.lo[k], std::nextafterf(mn, -inf));
                it.hi[k] = std::max(it.hi[k], std::nextafterf(mx, inf));
            }
        }
        return it;
    }
    Item8 link_item(int32_t link, const float *lo, const float *hi) const {
        Item8 it;
        if (link >= 0) {
            it.link = link;
            it.tb = it.te = 0;
        } else {  // binary leaf: its triangle run
            it.link = -1;
            it.tb = static_cast<uint32_t>(~link);
            it.te = it.tb;
            while (!(tris[it.te].id_last & RT_LAST_BIT)) ++it.te;
            ++it.te;
        }
        std::memcpy(it.lo, lo, 12);
        std::memcpy(it.hi, hi, 12);
        return it;
    }
    void open(const Item8 &it, Item8 two[2]) const {
        if (it.link >= 0) {
            const DNode &n = nodes[it.link];
            const float llo[3] = {n.lminx, n.lminy, n.lminz}, lhi[3] = {n.lmaxx, n.lmaxy, n.lmaxz};
            const float rlo[3] = {n.rminx, n.rminy, n.rminz}, rhi[3] = {n.rmaxx, n.rmaxy, n.rmaxz};
            two[0] = link_item(n.left, llo, lhi);
            two[1] = link_item(n.right, rlo, rhi);
        } else {  // a leaf of more than kLeaf8 triangles: halves (the run keeps its order)
            const uint32_t mid = it.tb + (it.te - it.tb + 1) / 2;
            two[0] = range_item(it.tb, mid);
            two[1] = range_item(mid, it.te);
        }
    }
    // Cost-optimal collapse (Ylitie, Karras & Laine 2017, sec. 4.1, without leaf merging): c[i-1] = the least summed box
    // area of the wide nodes below an item when it may occupy at most i slots of its parent; s[i-1] = slots given to
    // its first half (0: same as with i-1 slots; i == 1: the item is a wide node of its own and s[0] splits its 8 slots).
    struct Table {
        float c[8];
        uint8_t s[8];
    };
    std::vector<Table> memo;
    std::vector<uint8_t> memo_done;
    Table table_of(const Item8 &item) {  // item.openable()
        if (item.link >= 0 && memo_done[item.link]) return memo[item.link];
        Item8 two[2];
        open(item, two);
        Table t[2];
        bool op[2];
        for (int c = 0; c < 2; ++c) {
            op[c] = two[c].openable();
            if (op[c]) t[c] = table_of(two[c]);
        }
        float dist[9];
        uint8_t arg[9];
        for (int j = 2; j <= 8; ++j) {
            dist[j] = std::numeric_limits<float>::infinity();
            arg[j] = 1;
            for (int a = 1; a < j; ++a) {
                const float v = (op[0] ? t[0].c[std::min(a, 7) - 1] : 0.0f) + (op[1] ? t[1].c[std::min(j - a, 7) - 1] : 0.0f);
                if (v < dist[j]) {
                    dist[j] = v;
                    arg[j] = static_cast<uint8_t>(a);
                }
            }
        }
        Table r;
        r.c[0] = box_area(item) + dist[8];
        r.s[0] = arg[8];
        for (int i = 2; i <= 8; ++i) {
            if (dist[i] < r.c[i - 2]) {
                r.c[i - 1] = dist[i];
                r.s[i - 1] = arg[i];
            } else {
                r.c[i - 1] = r.c[i - 2];
                r.s[i - 1] = 0;
            }
        }
        if (item.link >= 0) {
            memo[item.link] = r;
            memo_done[item.link] = 1;
        }
        return r;
    }
    void expand(const Item8 &item, int slots, Item8 *out_items, int &n) {
        if (!item.openable()) {
            out_items[n++] = item;
            return;
        }
        const Table t = table_of(item);
        while (slots > 1 && t.s[slots - 1] == 0) --slots;
        if (slots == 1) {
            out_items[n++] = item;  // stays an inner child: a wide node of its own
            return;
        }
        const int a = t.s[slots - 1];
        Item8 two[2];
        open(item, two);
        expand(two[0], std::min(a, 7), out_items, n);
        expand(two[1], std::min(slots - a, 7), out_items, n);
    }
    // builds wide node `idx` (already allocated) from `self`
    void build(const Item8 &self, uint32_t idx) {
        Item8 it[8];
        int n = 0;
        if (!self.openable()) {
            it[n++] = self;
        } else if (RT_COLLAPSE8_OPTIMAL) {
            const Table t = table_of(self);
            Item8 two[2];
            open(self, two);
            expand(two[0], std::min<int>(t.s[0], 7), it, n);
            expand(two[1], std::min<int>(8 - t.s[0], 7), it, n);
        } else {
            open(self, it);
            n = 2;
            while (n < 8) {  // greedy: open the child with the largest box until eight children or nothing left to open
                int best = -1;
                float best_area = -1.0f;
                for (int i = 0; i < n; ++i)
                    if (it[i].openable() && box_area(it[i]) > best_area) {
                        best_area = box_area(it[i]);
                        best = i;
                    }
                if (best < 0) break;
                Item8 two[2];
                open(it[best], two);
                it[best] = two[0];
                it[n++] = two[1];
            }
        }
        // slots by octant: greedily the (child, slot) pair with the largest dot(child centre - node centre, slot direction)
        float c[3];
        for (int k = 0; k < 3; ++k) {
            float lo = it[0].lo[k], hi = it[0].hi[k];
            for (int i = 1; i < n; ++i) lo = std::min(lo, it[i].lo[k]), hi = std::max(hi, it[i].hi[k]);
            c[k] = 0.5f * (lo + hi);
        }
        int slot_of[8];
        bool used[8] = {false, false, false, false, false, false, false, false}, done[8] = {false, false, false, false, false, false, false, false};
        for (int round = 0; round < n; ++round) {
            float bestv = -std::numeric_limits<float>::infinity();
            int bi = -1, bs = -1;
            for (int i = 0; i < n; ++i) {
                if (done[i]) continue;
                for (int s = 0; s < 8; ++s) {
                    if (used[s]) continue;
                    float v = 0.0f;
                    for (int k = 0; k < 3; ++k) {
                        const float cc = 0.5f * (it[i].lo[k] + it[i].hi[k]) - c[k];
                        v += ((s >> k) & 1) ? cc : -cc;
                    }
                    if (v > bestv || bi < 0) bestv = v, bi = i, bs = s;
                }
            }
            done[bi] = true;
            used[bs] = true;
            slot_of[bi] = bs;
        }
        int item_in[8];
        for (int s = 0; s < 8; ++s) item_in[s] = -1;
        for (int i = 0; i < n; ++i) item_in[slot_of[i]] = i;
        QNode8 q;
        std::memset(&q, 0, sizeof q);
        Node8Boxes nb;
        std::memset(&nb, 0, sizeof nb);
        q.child_base = static_cast<uint32_t>(out.size());
        q.tri_base = static_cast<uint32_t>(perm.size());
        uint32_t n_inner = 0;
        for (int s = 0; s < 8; ++s) {
            const int i = item_in[s];
            if (i < 0) continue;
            nb.present |= static_cast<uint8_t>(1u << s);
            std::memcpy(nb.lo[s], it[i].lo, 12);
            std::memcpy(nb.hi[s], it[i].hi, 12);
            if (it[i].openable()) {
                q.imask |= 1u << s;
                ++n_inner;
            } else {
                q.counts |= (it[i].te - it[i].tb) << (2 * s);
                for (uint32_t t = it[i].tb; t < it[i].te; ++t) perm.push_back(t);
                last.push_back(static_cast<uint32_t>(perm.size() - 1));
            }
        }
        out.resize(out.size() + n_inner);
        boxes.resize(out.size());
        out[idx] = q;
        boxes[idx] = nb;
        uint32_t rank = 0;
        for (int s = 0; s < 8; ++s)
            if (q.imask >> s & 1u) build(it[item_in[s]], q.child_base + rank++);
    }
};
inline int quantize_nodes8(const std::vector<Node8Boxes> &boxes, std::vector<QNode8> &out) {
    std::atomic<int> rc{RT_OK};
    parallel_for(out.size(), [&](size_t b, size_t e) {
        for (size_t k = b; k < e; ++k) {
            const Node8Boxes &nb = boxes[k];
            QNode8 &q = out[k];
            for (int a = 0; a < 3; ++a) {
                float lo[8], hi[8];
                uint8_t ql[8], qh[8], fl[8], fh[8];
                int m = 0;
                for (int s = 0; s < 8; ++s)
                    if (nb.present >> s & 1) {
                        lo[m] = nb.lo[s][a];
                        hi[m] = nb.hi[s][a];
                        ++m;
                    }
                if (!quantize_axis_n(lo, hi, m, q.org[a], ql, qh)) rc = RT_ERR_BAD_SCENE;
                m = 0;
                for (int s = 0; s < 8; ++s) {
                    if (nb.present >> s & 1) {
                        fl[s] = ql[m];
                        fh[s] = qh[m];
                        ++m;
                    } else {  // empty slot: inverted box, never hit
                        fl[s] = 255;
                        fh[s] = 0;
                    }
                }
                auto word = [](const uint8_t *p) {
                    return static_cast<uint32_t>(p[0]) | static_cast<uint32_t>(p[1]) << 8 | static_cast<uint32_t>(p[2]) << 16 |
                           static_cast<uint32_t>(p[3]) << 24;
                };
                q.g0[a] = word(fl);
                q.g0[3 + a] = word(fh);
                q.g1[a] = word(fl + 4);
                q.g1[3 + a] = word(fh + 4);
            }
        }
    });
    return rc;
}

}  // namespace detail

// `formats`: which quantised node arrays to produce (the device build needs one, the host checks both)
// RT_PACK_Q8 re-orders the triangles, so it excludes the other two
enum { RT_PACK_Q2 = 1, RT_PACK_Q4 = 2, RT_PACK_ALL = 3, RT_PACK_Q8 = 4 };
// `built_tree`: src comes from sah_build.h (well formed), which allows the direct parallel 4-wide collapse
inline int pack_bvh(const rt_scene_desc &sc, const rt_bvh_desc &src, PackedBvh &out, int formats = RT_PACK_ALL, bool built_tree = false) {
    out.nodes.clear();
    out.tris.assign(src.n_objects, DTri());
    out.order.assign(src.objects, src.objects + src.n_objects);
    out.root = RT_LINK_NONE;
    out.root4 = RT_LINK_NONE;
    out.max_depth = 0;
    out.stack_need4 = 0;
    out.qnodes.clear();
    out.qnodes4.clear();
    out.qnodes8.clear();
    PackLap lap;
    detail::parallel_for(src.n_objects, [&](size_t kb, size_t ke) {
        for (size_t k = kb; k < ke; ++k) {
            const uint32_t id = src.objects[k];
            const float *p = sc.tri_pos + static_cast<size_t>(id) * 9;
            DTri &t = out.tris[k];
            t.ax = p[0]; t.ay = p[1]; t.az = p[2];
            t.e1x = p[3] - p[0]; t.e1y = p[4] - p[1]; t.e1z = p[5] - p[2];
            t.e2x = p[6] - p[0]; t.e2y = p[7] - p[1]; t.e2z = p[8] - p[2];
            t.pad0 = t.pad1 = 0.0f;
            t.pad2[0] = t.pad2[1] = t.pad2[2] = t.pad2[3] = 0.0f;
            t.id_last = id;
        }
    });
    if (src.root == RT_NO_CHILD || src.n_objects == 0) return RT_OK;
    if (built_tree && formats == RT_PACK_Q4) {
        DTri null_tri;
        std::memset(&null_tri, 0, sizeof null_tri);
        null_tri.id_last = RT_LAST_BIT;
        out.tris.push_back(null_tri);
        const int32_t null_leaf = ~static_cast<int32_t>(out.tris.size() - 1);
        std::vector<detail::Node4Boxes> boxes;
        out.qnodes4.reserve(src.n_nodes / 3 + 64);
        boxes.reserve(src.n_nodes / 3 + 64);
        lap.lap(1);
        out.root4 = detail::collapse4_built(src, out.tris, null_leaf, out.qnodes4, boxes);
        out.stack_need4 = detail::stack_need4(out.qnodes4, out.root4, null_leaf);
        if (out.stack_need4 > RT_EXT_STACK_CAP) return RT_ERR_BAD_SCENE;
        lap.lap(2);
        if (int rq = detail::quantize_nodes4(boxes, out.qnodes4)) return rq;
        lap.lap(3);
        return RT_OK;
    }
    int rc = RT_OK;
    out.root = detail::pack_node(src, src.root, out, 0, rc);
    if (rc) return rc;
    lap.lap(1);
    if (formats & RT_PACK_Q8) {
        if (formats != RT_PACK_Q8) return RT_ERR_INVALID_ARG;
        std::vector<detail::Node8Boxes> boxes;
        std::vector<uint32_t> perm, last;
        perm.reserve(src.n_objects);
        out.qnodes8.reserve(out.nodes.size() / 3 + 2);
        detail::Collapse8 cl{out.nodes, out.tris, out.qnodes8, boxes, perm, last, {}, {}};
        cl.memo.resize(out.nodes.size());
        cl.memo_done.assign(out.nodes.size(), 0);
        // root item: the box is not needed (the root's own box is never tested, bvh.h:170-180)
        const float z[3] = {0.0f, 0.0f, 0.0f};
        detail::Item8 root = cl.link_item(out.root, z, z);
        if (root.link < 0) root = cl.range_item(root.tb, root.te);  // ... unless the root is a leaf: its box is a child box
        out.qnodes8.emplace_back();
        boxes.emplace_back();
        cl.build(root, 0);
        if (perm.size() != src.n_objects) return RT_ERR_BAD_SCENE;
        if (int rq = detail::quantize_nodes8(boxes, out.qnodes8)) return rq;
        std::vector<DTri> nt(src.n_objects);
        std::vector<uint32_t> no(src.n_objects);
        for (uint32_t k = 0; k < src.n_objects; ++k) {
            nt[k] = out.tris[perm[k]];
            nt[k].id_last &= ~RT_LAST_BIT;
            no[k] = out.order[perm[k]];
        }
        for (uint32_t k : last) nt[k].id_last |= RT_LAST_BIT;
        out.tris.swap(nt);
        out.order.swap(no);
        out.nodes.clear();  // their leaf links refer to the old triangle order
        out.root = RT_LINK_NONE;
        DTri null_tri;  // pair loads of the leaf phase may read one triangle past a leaf
        std::memset(&null_tri, 0, sizeof null_tri);
        null_tri.id_last = RT_LAST_BIT;
        out.tris.push_back(null_tri);
        return RT_OK;
    }
    if (formats & RT_PACK_Q2)
        if (int rq = detail::quantize_nodes(out.nodes, out.qnodes)) return rq;
    // 4-wide collapse; the null leaf (absent children) is one degenerate triangle appended after the real ones
    out.qnodes4.clear();
    DTri null_tri;
    std::memset(&null_tri, 0, sizeof null_tri);
    null_tri.id_last = RT_LAST_BIT;
    out.tris.push_back(null_tri);
    if (formats & RT_PACK_Q4) {
        const int32_t null_leaf = ~static_cast<int32_t>(out.tris.size() - 1);
        std::vector<detail::Node4Boxes> boxes;
        out.qnodes4.reserve(out.nodes.size() / 2 + 1);
        boxes.reserve(out.nodes.size() / 2 + 1);
        out.root4 = detail::collapse4(out.nodes, out.root, null_leaf, out.qnodes4, boxes);
        out.stack_need4 = detail::stack_need4(out.qnodes4, out.root4, null_leaf);
        if (out.stack_need4 > RT_EXT_STACK_CAP) return RT_ERR_BAD_SCENE;
        lap.lap(2);
        if (int rq = detail::quantize_nodes4(boxes, out.qnodes4)) return rq;
        lap.lap(3);
    }
    return rc;
}

// The light side of a scene: out.light (the light BVH; the traversal of the all-hit light pdf uses a rebuilt tree when
// `rebuild`), out.light_sample (the sampling list, in the host light BVH's object order) and out.light_extra (DLight
// normals and areas).  Reads sc.tri_pos and sc.light_bvh only, so that rt_gpu_update_geometry can run it on new positions.
inline int pack_lights(const rt_scene_desc &sc, PackedScene &out, bool rebuild, int formats) {
    PackedBvh host_order;
    if (int rc = pack_bvh(sc, sc.light_bvh, host_order, formats == RT_PACK_Q8 ? 0 : formats)) return rc;
    out.light_sample = host_order.tris;
    if (formats == RT_PACK_Q8 && !(rebuild && sc.light_bvh.n_objects > 0 && sc.light_bvh.root != RT_NO_CHILD)) {
        if (int rc = pack_bvh(sc, sc.light_bvh, out.light, formats)) return rc;
    } else if (rebuild && sc.light_bvh.n_objects > 0 && sc.light_bvh.root != RT_NO_CHILD) {
        BuiltBvh built;
        build_sah_bvh(sc.tri_pos, sc.light_bvh.objects, sc.light_bvh.n_objects, built);
        if (int rc = pack_bvh(sc, built.desc(), out.light, formats, true)) return rc;
    } else {
        out.light = host_order;
    }
    out.light_extra.resize(sc.light_bvh.n_objects);
    for (uint32_t k = 0; k < sc.light_bvh.n_objects; ++k) {
        const DTri &t = out.light.tris[k];
        // crs(v, u), triangle::normal / square (geometry.h:477-483)
        const float cx = t.e1y * t.e2z - t.e1z * t.e2y;
        const float cy = t.e1z * t.e2x - t.e1x * t.e2z;
        const float cz = t.e1x * t.e2y - t.e1y * t.e2x;
        const float l = std::sqrt(cx * cx + cy * cy + cz * cz);
        out.light_extra[k] = {cx / l, cy / l, cz / l, l / 2};
    }
    return RT_OK;
}

// `rebuild_scene_bvh`: build the scene BVH with the library's SAH builder (sah_build.h) over the triangles of
// sc.scene_bvh instead of adopting the host's tree; the light BVH is always adopted as passed.
// A host that passes NO scene BVH (scene_bvh.n_nodes == 0; rt_gpu.h) leaves the build to the library: the tree is built
// over all n_tris triangles in scene.objects order.
// `with_scene` = false: only the small host-side parts (light BVH, sampling list, materials, textures, LUT); the scene BVH,
// triangles and attributes are then produced on the device (gpu_build.cuh).
inline int pack_scene(const rt_scene_desc &sc, PackedScene &out, bool rebuild_scene_bvh = false, int formats = RT_PACK_ALL,
                      bool with_scene = true) {
    PackLap lap;
    const bool no_host_tree = sc.scene_bvh.n_nodes == 0 && sc.n_tris > 0;
    if (!with_scene) {
        out.scene = PackedBvh();
    } else if (no_host_tree) {
        build_sah_bvh(sc.tri_pos, nullptr, sc.n_tris, out.built, &out.sah_scratch);
        lap.lap(0);
        if (int rc = pack_bvh(sc, out.built.desc(), out.scene, formats, true)) return rc;
    } else if (rebuild_scene_bvh && sc.scene_bvh.n_objects > 0 && sc.scene_bvh.root != RT_NO_CHILD) {
        build_sah_bvh(sc.tri_pos, sc.scene_bvh.objects, sc.scene_bvh.n_objects, out.built, &out.sah_scratch);
        lap.lap(0);
        if (int rc = pack_bvh(sc, out.built.desc(), out.scene, formats, true)) return rc;
    } else if (int rc = pack_bvh(sc, sc.scene_bvh, out.scene, formats)) {
        return rc;
    }
    if (int rc = pack_lights(sc, out, rebuild_scene_bvh, formats)) return rc;

    lap = PackLap();
    const uint32_t n = with_scene ? static_cast<uint32_t>(out.scene.order.size()) : 0u;  // device triangle order = packed BVH order
    out.attrs.resize(n);
    bool any_tangent = false;
    if (sc.tri_tangents && with_scene)
        for (size_t i = 0; i < static_cast<size_t>(sc.n_tris) * 3 && !any_tangent; ++i) {
            const float *t = sc.tri_tangents + i * 3;
            any_tangent = !(t[0] == 1.0f && t[1] == 0.0f && t[2] == 0.0f);
        }
    out.tangents.clear();
    if (any_tangent) out.tangents.resize(n);
    detail::parallel_for(n, [&](size_t kb, size_t ke) {
        for (size_t k = kb; k < ke; ++k) {
            const uint32_t id = out.scene.order[k];
            const float *nn = sc.tri_normals + static_cast<size_t>(id) * 9;
            const float *uv = sc.tri_uv + static_cast<size_t>(id) * 6;
            DAttr &a = out.attrs[k];
            a.n0x = nn[0]; a.n0y = nn[1]; a.n0z = nn[2];
            a.n1x = nn[3]; a.n1y = nn[4]; a.n1z = nn[5];
            a.n2x = nn[6]; a.n2y = nn[7]; a.n2z = nn[8];
            a.uv0x = uv[0]; a.uv0y = uv[1]; a.uv1x = uv[2]; a.uv1y = uv[3]; a.uv2x = uv[4]; a.uv2y = uv[5];
            a.material = sc.tri_material[id];
            if (any_tangent) {
                const float *t = sc.tri_tangents + static_cast<size_t>(id) * 9;
                DTangent &d = out.tangents[k];
                d.t0x = t[0]; d.t0y = t[1]; d.t0z = t[2];
                d.t1x = t[3]; d.t1y = t[4]; d.t1z = t[5];
                d.t2x = t[6]; d.t2y = t[7]; d.t2z = t[8];
                d.pad0 = d.pad1 = d.pad2 = 0.0f;
            }
        }
    });
    lap.lap(5);

    out.materials.resize(sc.n_materials);
    for (uint32_t i = 0; i < sc.n_materials; ++i) {
        const rt_material &m = sc.materials[i];
        DMat &d = out.materials[i];
        std::memcpy(d.color, m.color, sizeof d.color);
        std::memcpy(d.emission, m.emission, sizeof d.emission);
        d.roughness = m.roughness;
        d.metallic = m.metallic;
        d.ior = m.ior;
        d.color_tex = m.color_tex;
        d.emissive_tex = m.emissive_tex;
        d.mr_tex = m.metallic_roughness_tex;
        d.normal_tex = m.normal_tex;
        d.pad0 = d.pad1 = 0;
    }

    out.textures.resize(sc.n_textures);
    out.texels.resize(sc.texel_bytes / 4);
    if (sc.texel_bytes) std::memcpy(out.texels.data(), sc.texels, out.texels.size() * 4);
    for (uint32_t i = 0; i < sc.n_textures; ++i) {
        if (sc.textures[i].offset % 4) return RT_ERR_BAD_SCENE;
        out.textures[i] = {static_cast<uint32_t>(sc.textures[i].offset / 4), sc.textures[i].width,
                           sc.textures[i].height, 0};
    }
    for (int k = 0; k < 256; ++k) out.gamma_lut[k] = std::pow(static_cast<float>(k) / 255.0f, 2.2f);
    lap.lap(6);
    return RT_OK;
}

// Fill the pointer-free part of a DScene; pointers are set by the caller (device or host arrays).
inline void fill_scene_constants(const rt_scene_desc &sc, const PackedScene &p, DScene &d) {
    std::memset(&d, 0, sizeof d);
    d.scene.root = p.scene.root;
    d.scene.root4 = p.scene.root4;
    d.light.root4 = p.light.root4;
    d.scene.n_nodes8 = static_cast<uint32_t>(p.scene.qnodes8.size());
    d.light.n_nodes8 = static_cast<uint32_t>(p.light.qnodes8.size());
    d.scene.n_tris = static_cast<uint32_t>(p.scene.tris.size());
    d.light.root = p.light.root;
    d.light.n_tris = static_cast<uint32_t>(p.light.tris.size());
    d.n_lights = sc.light_bvh.n_objects;
    d.ray_depth = sc.ray_depth;
    d.eps = sc.eps;
    d.min_roughness = sc.min_roughness;
    d.vndf_factor = sc.vndf_factor;
    for (int k = 0; k < 3; ++k) {
        d.bg[k] = sc.bg_color[k];
        d.cam_pos[k] = sc.camera.position[k];
        d.cam_right[k] = sc.camera.right[k];
        d.cam_up[k] = sc.camera.up[k];
        d.cam_fwd[k] = sc.camera.forward[k];
    }
    d.fov_x = sc.camera.fov_x;
    d.env_tex = static_cast<int32_t>(sc.env_texture) - 1;  // 0 = constant sky
}

}  // namespace rt

#endif  // RT_REPACK_H
