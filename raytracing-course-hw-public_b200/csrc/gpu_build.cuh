// gpu_build.cuh — the scene preparation of rt_gpu_upload_scene on the DEVICE (SURVEY.md 8(f)-2: "BVH build on GPU
// replacing BVH::build", src/bvh.h:262-393).  Input: the host's per-triangle arrays exactly as rt_scene_desc passes
// them (copied H2D once); output: everything k_extend / k_shade read — QNode4 nodes, DTri, DAttr (, DTangent).
//
//   kb_setup        per triangle: box; scene box + centroid box (warp reduce + ordered-uint atomics)
//   big phase       level-synchronous binned SAH over the nodes with more than kSmall triangles (32 bins x 3 axes,
//                   the cost function and decisions of sah_build.h): kb_bin (one thread per triangle, atomics into
//                   the node's bins), kb_split (one thread per node: sweep, children), kb_flags / kb_scan /
//                   kb_scatter (stable partition by prefix sums: the result does not depend on scheduling)
//   kb_small        one WARP per node of <= kSmall triangles builds its whole sub-tree in shared memory (8 bins,
//                   one candidate split per lane)
//   kb_tris/attrs   DTri / DAttr / DTangent in BVH order
//   collapse        kb_mark (top-down, one launch per wide level: which binary nodes become 4-wide nodes, worst-case
//                   traversal-stack need), kb_markwords + kb_scan (their numbering), kb_emit (children, quantisation)
//
// The binary tree uses the node slots of sah_build.h (left child = slot + 1, right child = slot + 2 * n_left), so no
// allocation is needed and the numbering is deterministic; the light BVH (a few dozen triangles) stays on the host.
// Everything is plain CUDA-core integer / float work bound by launch latency and L2 atomics: ~2-3 ms for 260k triangles
// against 17 ms (16 host threads) for the same algorithm in sah_build.h.
#ifndef RT_GPU_BUILD_CUH
#define RT_GPU_BUILD_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#include "quantize.h"
#include "rt_gpu.h"
#include "rt_types.h"

namespace rtb {

constexpr uint32_t kSmall = 32;    // nodes of at most this many triangles are finished by one warp (kb_small)
constexpr int kBins = 32;          // sah_build.h: kBins
constexpr int kSmallBins = 8;      // sah_build.h: nb for n <= 32
constexpr uint32_t kMaxLeaf = 8;   // sah_build.h: kMaxLeaf
constexpr float kTraversalCost = 1.0f;
constexpr uint32_t kNoLevel = 0xFFFFFFFFu;
constexpr uint32_t kOrdPosInf = 0xFF800000u;  // f2ord(+inf)
constexpr uint32_t kOrdNegInf = 0x007FFFFFu;  // f2ord(-inf)

// order-preserving float <-> uint32 map, so that atomicMin / atomicMax on the integers are min / max of the floats
__device__ __forceinline__ uint32_t f2ord(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u); }

struct Counters {
    uint32_t n_active[2];   // big nodes of the current / next level
    uint32_t n_small;       // nodes handed to kb_small
    uint32_t max_depth;     // of the binary tree
    uint32_t error;         // bit 0: non-finite geometry / node that cannot be quantised
    uint32_t any_tangent;   // some tangent differs from (1,0,0)
    uint32_t frontier[3];   // wide roots of the collapse levels l, l + 1 (being filled), l + 2 (being cleared), modulo 3
    uint32_t stack_need;    // worst-case traversal-stack entries of the 4-wide tree
    uint32_t n_wide;        // 4-wide nodes
    uint32_t root_box[6];   // ordered: scene box lo, hi
    uint32_t root_cb[6];    // ordered: centroid box lo, hi
    uint32_t pad[9];
};

// per binary-node slot, while the tree is being built
struct alignas(16) NodeAux {
    float cbl[3], cbh[3];   // centroid box
    float scale[3];         // bins / centroid extent per axis (0: axis not usable)
    uint32_t begin, count;  // triangle positions [begin, begin + count)
    uint32_t level;         // big-phase level at which this node is binned and split (kNoLevel: never)
    uint32_t binslot;       // its bins in the pool of that level
    uint32_t depth;
    int32_t axis;           // decided split: 0..2 binned, 3 by index
    uint32_t bin;           // last bin of the left side
    uint32_t nleft;
    uint32_t pad[3];
};

struct BinSlot {  // 32 bins x 3 axes: count, triangle-box union, centroid-box union (ordered uints)
    uint32_t cnt[3][kBins];
    uint32_t blo[3][kBins][3], bhi[3][kBins][3];
    uint32_t clo[3][kBins][3], chi[3][kBins][3];
};

struct Box {
    float lo[3], hi[3];
    __device__ void reset() {
        for (int k = 0; k < 3; ++k) {
            lo[k] = HUGE_VALF;
            hi[k] = -HUGE_VALF;
        }
    }
    __device__ void grow(const float *l, const float *h) {
        for (int k = 0; k < 3; ++k) {
            lo[k] = l[k] < lo[k] ? l[k] : lo[k];
            hi[k] = h[k] > hi[k] ? h[k] : hi[k];
        }
    }
    __device__ float area() const {  // sah_build.h Box3::area, same operation order
        const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        return __fadd_rn(__fadd_rn(__fmul_rn(dx, dy), __fmul_rn(dy, dz)), __fmul_rn(dz, dx));
    }
};

__device__ __forceinline__ int bin_of(float c, float cmin, float scale, int nb) {
    int k = static_cast<int>(__fmul_rn(__fsub_rn(c, cmin), scale));
    return k < 0 ? 0 : (k >= nb ? nb - 1 : k);
}

struct Arrays {
    // inputs (scene.objects order)
    const float *tri_pos, *tri_normals, *tri_uv, *tri_tangents;
    const uint32_t *tri_material;
    uint32_t n;
    // build state
    float4 *plo, *phi;            // [n] triangle boxes
    uint32_t *idx[2];             // [n] triangle at each position (ping-pong)
    uint32_t *node_of[2];         // [n] node slot of each position
    rt_bvh_node *nodes;           // [2n-1] the binary tree, sah_build.h's slot layout
    NodeAux *aux;                 // [2n-1]
    BinSlot *bins[2];             // [n / kSmall + 1] per level parity
    uint32_t *active[2];          // big nodes of a level
    uint32_t *small;              // nodes for kb_small
    uint32_t *words, *wscan;      // ballot words of a flag array and the exclusive scan of their popcounts
    uint8_t *last;                // [n] position ends a leaf
    uint8_t *mark;                // [2n-1] binary node is the root of a 4-wide node
    uint32_t *need;               // [2n-1] traversal-stack entries above that wide node
    uint32_t *frontier[3];
    Counters *c;
    // outputs
    QNode4 *qnodes4;
    DTri *tris;                   // [n + 1] BVH order + the null triangle
    DAttr *attrs;                 // [n]
    DTangent *tangents;           // [n] or null
};

// ---- setup ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_minmax_atomic(uint32_t *lo3_hi3, const float lo[3], const float hi[3]) {
    float v[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]};
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const float o = __shfl_xor_sync(0xFFFFFFFFu, v[k], off);
            v[k] = k < 3 ? fminf(v[k], o) : fmaxf(v[k], o);
        }
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 3; ++k) atomicMin(lo3_hi3 + k, f2ord(v[k]));
        for (int k = 3; k < 6; ++k) atomicMax(lo3_hi3 + k, f2ord(v[k]));
    }
}

__global__ void __launch_bounds__(256) kb_init(Arrays A) {
    Counters &c = *A.c;
    c.n_active[0] = c.n_active[1] = c.n_small = c.max_depth = c.error = c.any_tangent = 0;
    c.frontier[0] = c.frontier[1] = c.frontier[2] = c.stack_need = c.n_wide = 0;
    for (int k = 0; k < 3; ++k) {
        c.root_box[k] = c.root_cb[k] = kOrdPosInf;
        c.root_box[3 + k] = c.root_cb[3 + k] = kOrdNegInf;
    }
}

__global__ void __launch_bounds__(256) kb_setup(Arrays A) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = {HUGE_VALF, HUGE_VALF, HUGE_VALF}, hi[3] = {-HUGE_VALF, -HUGE_VALF, -HUGE_VALF};
    float cl[3] = {HUGE_VALF, HUGE_VALF, HUGE_VALF}, ch[3] = {-HUGE_VALF, -HUGE_VALF, -HUGE_VALF};
    if (i < A.n) {
        const float *p = A.tri_pos + static_cast<size_t>(i) * 9;
        bool finite = true;
        for (int k = 0; k < 3; ++k) {
            const float a = p[k], b = p[3 + k], c = p[6 + k];
            lo[k] = fminf(a, fminf(b, c));
            hi[k] = fmaxf(a, fmaxf(b, c));
            finite = finite && rt::detail::finite_f(a) && rt::detail::finite_f(b) && rt::detail::finite_f(c);
            cl[k] = ch[k] = __fmul_rn(0.5f, __fadd_rn(lo[k], hi[k]));
        }
        if (!finite) atomicOr(&A.c->error, 1u);
        A.plo[i] = make_float4(lo[0], lo[1], lo[2], 0.0f);
        A.phi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
        A.idx[0][i] = i;
        A.node_of[0][i] = 0;
        A.last[i] = 0;
    }
    warp_minmax_atomic(A.c->root_box, lo, hi);
    warp_minmax_atomic(A.c->root_cb, cl, ch);
}

// does any tangent differ from the loader's default (1,0,0)?  (The reference's loader never finds a tangent attribute,
// scene.h:336, so hosts pass n x 9 default floats; DTangent is only built when it matters.)
__global__ void __launch_bounds__(256) kb_tangent_flag(Arrays A) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool tangent = false;
    if (i < A.n && A.tri_tangents) {
        const float *t = A.tri_tangents + static_cast<size_t>(i) * 9;
        for (int v = 0; v < 3; ++v) tangent = tangent || !(t[v * 3] == 1.0f && t[v * 3 + 1] == 0.0f && t[v * 3 + 2] == 0.0f);
    }
    if (__any_sync(0xFFFFFFFFu, tangent) && (threadIdx.x & 31) == 0) atomicOr(&A.c->any_tangent, 1u);
}

// a freshly created node: record, and its place in the next level's work lists.  Called by a whole warp (lane 0 writes
// the records, all lanes clear the node's bins).
__device__ void open_node(Arrays &A, uint32_t slot, uint32_t begin, uint32_t count, uint32_t depth, const Box &box, const Box &cb,
                          uint32_t next_level, int next_parity) {
    const int lane = threadIdx.x & 31;
    uint32_t k = 0;
    if (lane == 0) {
        rt_bvh_node &nd = A.nodes[slot];
        for (int d = 0; d < 3; ++d) {
            nd.bmin[d] = box.lo[d];
            nd.bmax[d] = box.hi[d];
        }
        nd.left_child = nd.right_child = RT_NO_CHILD;
        nd.obj_begin = nd.obj_end = 0;
        NodeAux &x = A.aux[slot];
        for (int d = 0; d < 3; ++d) {
            x.cbl[d] = cb.lo[d];
            x.cbh[d] = cb.hi[d];
            const float ext = __fsub_rn(cb.hi[d], cb.lo[d]);
            x.scale[d] = ext > 0.0f ? __fdiv_rn(static_cast<float>(kBins), ext) : 0.0f;
        }
        x.begin = begin;
        x.count = count;
        x.depth = depth;
        x.axis = -1;
        x.bin = x.nleft = 0;
        x.level = kNoLevel;
        x.binslot = 0;
        atomicMax(&A.c->max_depth, depth);
        if (count > kSmall) {
            k = atomicAdd(&A.c->n_active[next_parity], 1u);
            A.active[next_parity][k] = slot;
            x.level = next_level;
            x.binslot = k;
        } else {
            A.small[atomicAdd(&A.c->n_small, 1u)] = slot;
        }
    }
    k = __shfl_sync(0xFFFFFFFFu, k, 0);
    if (count > kSmall) {
        uint32_t *g = reinterpret_cast<uint32_t *>(&A.bins[next_parity][k]);
        constexpr uint32_t kWords = sizeof(BinSlot) / 4, kCnt = 3 * kBins, kBox = 9 * kBins;
        for (uint32_t w = lane; w < kWords; w += 32)
            g[w] = w < kCnt ? 0u : (((w - kCnt) / kBox) & 1u ? kOrdNegInf : kOrdPosInf);  // cnt | blo | bhi | clo | chi
    }
}

__global__ void kb_root(Arrays A) {  // one warp
    Box box, cb;
    for (int k = 0; k < 3; ++k) {
        box.lo[k] = ord2f(A.c->root_box[k]);
        box.hi[k] = ord2f(A.c->root_box[3 + k]);
        cb.lo[k] = ord2f(A.c->root_cb[k]);
        cb.hi[k] = ord2f(A.c->root_cb[3 + k]);
    }
    open_node(A, 0, 0, A.n, 0, box, cb, 0, 0);
}

// ---- big phase -----------------------------------------------------------------------------------------------------
// One thread per triangle position.  The positions of a node are contiguous, so a block whose first and last position
// lie in the same node belongs to that node entirely: it bins into shared memory and flushes the non-empty bins with one
// global atomic per word (the top levels, where a few nodes hold all triangles, would otherwise serialise 39 atomics
// per triangle on a few hundred addresses: 0.9 ms for the root level of 260k triangles, measured).  Blocks that straddle
// nodes (deep levels: many small nodes, little contention) go to the global bins directly.
__global__ void __launch_bounds__(256) kb_bin(Arrays A, uint32_t level, int parity) {
    __shared__ uint32_t s_bins[sizeof(BinSlot) / 4];
    const uint32_t p0 = blockIdx.x * blockDim.x, p = p0 + threadIdx.x;
    const uint32_t p_last = min(p0 + blockDim.x, A.n) - 1u;
    const uint32_t slot_first = A.node_of[parity][p0], slot_last = A.node_of[parity][p_last];
    const bool uniform = slot_first == slot_last;
    if (uniform && A.aux[slot_first].level != level) return;  // whole block in a node that is not split at this level
    constexpr uint32_t kWords = sizeof(BinSlot) / 4, kCnt = 3 * kBins, kBox = 9 * kBins;
    if (uniform) {
        for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x)
            s_bins[w] = w < kCnt ? 0u : (((w - kCnt) / kBox) & 1u ? kOrdNegInf : kOrdPosInf);  // cnt | blo | bhi | clo | chi
        __syncthreads();
    }
    if (p < A.n) {
        const uint32_t slot = A.node_of[parity][p];
        const NodeAux &x = A.aux[slot];
        if (x.level == level) {
            const uint32_t prim = A.idx[parity][p];
            const float4 l4 = A.plo[prim], h4 = A.phi[prim];
            const float lo[3] = {l4.x, l4.y, l4.z}, hi[3] = {h4.x, h4.y, h4.z};
            uint32_t olo[3], ohi[3], oc[3];
            float c[3];
            for (int k = 0; k < 3; ++k) {
                c[k] = __fmul_rn(0.5f, __fadd_rn(lo[k], hi[k]));
                olo[k] = f2ord(lo[k]);
                ohi[k] = f2ord(hi[k]);
                oc[k] = f2ord(c[k]);
            }
            BinSlot &b = uniform ? *reinterpret_cast<BinSlot *>(s_bins) : A.bins[level & 1][x.binslot];
            for (int a = 0; a < 3; ++a) {
                if (!(x.scale[a] > 0.0f)) continue;
                const int k = bin_of(c[a], x.cbl[a], x.scale[a], kBins);
                atomicAdd(&b.cnt[a][k], 1u);
                for (int d = 0; d < 3; ++d) {
                    atomicMin(&b.blo[a][k][d], olo[d]);
                    atomicMax(&b.bhi[a][k][d], ohi[d]);
                    atomicMin(&b.clo[a][k][d], oc[d]);
                    atomicMax(&b.chi[a][k][d], oc[d]);
                }
            }
        }
    }
    if (uniform) {
        __syncthreads();
        uint32_t *g = reinterpret_cast<uint32_t *>(&A.bins[level & 1][A.aux[slot_first].binslot]);
        for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) {
            const uint32_t v = s_bins[w];
            if (w < kCnt) {
                if (v) atomicAdd(g + w, v);
            } else if (((w - kCnt) / kBox) & 1u) {
                if (v != kOrdNegInf) atomicMax(g + w, v);
            } else if (v != kOrdPosInf) {
                atomicMin(g + w, v);
            }
        }
    }
}

__device__ __forceinline__ void load_box(const uint32_t lo[3], const uint32_t hi[3], float *l, float *h) {
    for (int k = 0; k < 3; ++k) {
        l[k] = ord2f(lo[k]);
        h[k] = ord2f(hi[k]);
    }
}

__device__ __forceinline__ int ceil_log2(uint32_t n) {
    int l = 0;
    while ((1u << l) < n) ++l;
    return l;
}

// warp-wide helpers of kb_split: lane = bin
struct LaneBox {
    float lo[3], hi[3];
    uint32_t cnt;
};
__device__ __forceinline__ LaneBox lane_merge(const LaneBox &a, const LaneBox &b) {
    LaneBox r;
    for (int k = 0; k < 3; ++k) {
        r.lo[k] = fminf(a.lo[k], b.lo[k]);
        r.hi[k] = fmaxf(a.hi[k], b.hi[k]);
    }
    r.cnt = a.cnt + b.cnt;
    return r;
}
__device__ __forceinline__ LaneBox lane_shfl(const LaneBox &v, int src) {
    LaneBox r;
    for (int k = 0; k < 3; ++k) {
        r.lo[k] = __shfl_sync(0xFFFFFFFFu, v.lo[k], src);
        r.hi[k] = __shfl_sync(0xFFFFFFFFu, v.hi[k], src);
    }
    r.cnt = __shfl_sync(0xFFFFFFFFu, v.cnt, src);
    return r;
}
// inclusive scan over the lanes: towards higher lanes (prefix) or towards lower lanes (suffix)
__device__ __forceinline__ LaneBox lane_scan(LaneBox v, bool suffix) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int src = suffix ? lane + off : lane - off;
        const LaneBox o = lane_shfl(v, (src < 0 || src > 31) ? lane : src);
        if (src >= 0 && src <= 31) v = lane_merge(v, o);
    }
    return v;
}
__device__ __forceinline__ float lane_area(const LaneBox &b) {  // sah_build.h Box3::area
    const float dx = b.hi[0] - b.lo[0], dy = b.hi[1] - b.lo[1], dz = b.hi[2] - b.lo[2];
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dy), __fmul_rn(dy, dz)), __fmul_rn(dz, dx));
}
__device__ __forceinline__ LaneBox lane_load(const uint32_t *cnt, const uint32_t (*lo)[3], const uint32_t (*hi)[3], int lane) {
    LaneBox v;
    v.cnt = cnt ? cnt[lane] : 0u;
    for (int k = 0; k < 3; ++k) {
        v.lo[k] = ord2f(lo[lane][k]);
        v.hi[k] = ord2f(hi[lane][k]);
    }
    return v;
}

// One WARP per node of the level, lane = bin: the serial sweep of sah_build.h becomes a prefix and a suffix scan over the
// lanes per axis (one thread per node spent ~0.15 ms per level in 190 dependent bin loads, whatever the node count).
__global__ void __launch_bounds__(128) kb_split(Arrays A, uint32_t level) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const int parity = level & 1;
    const int lane = threadIdx.x & 31;
    const uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (k >= A.c->n_active[parity]) return;
    const uint32_t slot = A.active[parity][k];
    NodeAux &x = A.aux[slot];
    const BinSlot &b = A.bins[parity][k];
    const uint32_t n = x.count;
    // depth budget (sah_build.h: force_median): an index-split tree over n triangles is ceil(log2 n) deep
    const bool force = static_cast<int>(x.depth) + ceil_log2(n) + 2 >= RT_STACK_SIZE - 2;
    float best_cost = HUGE_VALF;
    int best_key = 0x7FFFFFFF;  // axis * 32 + bin: the serial sweep keeps the first minimum in this order
    if (!force) {
        for (int axis = 0; axis < 3; ++axis) {
            if (!(x.scale[axis] > 0.0f)) continue;  // warp-uniform
            const LaneBox mine = lane_load(b.cnt[axis], b.blo[axis], b.bhi[axis], lane);
            const LaneBox pre = lane_scan(mine, false);   // bins 0 .. lane
            const LaneBox suf = lane_scan(mine, true);    // bins lane .. 31
            const LaneBox right = lane_shfl(suf, lane < 31 ? lane + 1 : 31);  // bins lane+1 .. 31
            if (lane < kBins - 1 && pre.cnt != 0 && right.cnt != 0) {  // split after bin `lane`
                const float cost = __fadd_rn(__fmul_rn(static_cast<float>(pre.cnt), lane_area(pre)),
                                             __fmul_rn(static_cast<float>(right.cnt), lane_area(right)));
                if (cost < best_cost) {
                    best_cost = cost;
                    best_key = axis * 32 + lane;
                }
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float oc = __shfl_xor_sync(FULL, best_cost, off);
            const int ok = __shfl_xor_sync(FULL, best_key, off);
            if (oc < best_cost || (oc == best_cost && ok < best_key)) {
                best_cost = oc;
                best_key = ok;
            }
        }
    }
    Box lb, rb, lc, rc;
    uint32_t nleft = 0;
    if (best_key != 0x7FFFFFFF) {  // n > kSmall >= kMaxLeaf: a node of the big phase is always split
        const int axis = best_key >> 5, bin = best_key & 31;
        const LaneBox tb = lane_load(b.cnt[axis], b.blo[axis], b.bhi[axis], lane);
        const LaneBox cb = lane_load(nullptr, b.clo[axis], b.chi[axis], lane);
        const LaneBox tl = lane_shfl(lane_scan(tb, false), bin), tr = lane_shfl(lane_scan(tb, true), bin + 1);
        const LaneBox cl = lane_shfl(lane_scan(cb, false), bin), cr = lane_shfl(lane_scan(cb, true), bin + 1);
        for (int d = 0; d < 3; ++d) {
            lb.lo[d] = tl.lo[d]; lb.hi[d] = tl.hi[d];
            rb.lo[d] = tr.lo[d]; rb.hi[d] = tr.hi[d];
            lc.lo[d] = cl.lo[d]; lc.hi[d] = cl.hi[d];
            rc.lo[d] = cr.lo[d]; rc.hi[d] = cr.hi[d];
        }
        nleft = tl.cnt;
        if (lane == 0) {
            x.axis = axis;
            x.bin = static_cast<uint32_t>(bin);
        }
    } else {  // all centroids coincide (or the depth budget is nearly used): split by position, boxes by a pass over the range
        nleft = n / 2;
        float v[24];
        for (int d = 0; d < 24; ++d) v[d] = (d % 6) < 3 ? HUGE_VALF : -HUGE_VALF;  // lb, lc, rb, rc as (lo3, hi3)
        const uint32_t *idx = A.idx[parity];
        for (uint32_t q = lane; q < n; q += 32) {
            const uint32_t prim = idx[x.begin + q];
            const float4 l4 = A.plo[prim], h4 = A.phi[prim];
            const float l[3] = {l4.x, l4.y, l4.z}, h[3] = {h4.x, h4.y, h4.z};
            const int o = q < nleft ? 0 : 12;
            for (int d = 0; d < 3; ++d) {
                const float c = __fmul_rn(0.5f, __fadd_rn(l[d], h[d]));
                v[o + d] = fminf(v[o + d], l[d]);
                v[o + 3 + d] = fmaxf(v[o + 3 + d], h[d]);
                v[o + 6 + d] = fminf(v[o + 6 + d], c);
                v[o + 9 + d] = fmaxf(v[o + 9 + d], c);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1)
#pragma unroll
            for (int d = 0; d < 24; ++d) {
                const float o = __shfl_xor_sync(FULL, v[d], off);
                v[d] = (d % 6) < 3 ? fminf(v[d], o) : fmaxf(v[d], o);
            }
        for (int d = 0; d < 3; ++d) {
            lb.lo[d] = v[d]; lb.hi[d] = v[3 + d];
            lc.lo[d] = v[6 + d]; lc.hi[d] = v[9 + d];
            rb.lo[d] = v[12 + d]; rb.hi[d] = v[15 + d];
            rc.lo[d] = v[18 + d]; rc.hi[d] = v[21 + d];
        }
        if (lane == 0) {
            x.axis = 3;
            x.bin = 0;
        }
    }
    const uint32_t lslot = slot + 1, rslot = slot + 2 * nleft;
    if (lane == 0) {
        x.nleft = nleft;
        rt_bvh_node &nd = A.nodes[slot];
        nd.left_child = lslot;
        nd.right_child = rslot;
    }
    open_node(A, lslot, x.begin, nleft, x.depth + 1, lb, lc, level + 1, parity ^ 1);
    open_node(A, rslot, x.begin + nleft, n - nleft, x.depth + 1, rb, rc, level + 1, parity ^ 1);
}

__device__ __forceinline__ bool goes_left(const Arrays &A, const NodeAux &x, uint32_t p, uint32_t prim) {
    if (x.axis == 3) return p - x.begin < x.nleft;
    const float4 l4 = A.plo[prim], h4 = A.phi[prim];
    const float lo = x.axis == 0 ? l4.x : (x.axis == 1 ? l4.y : l4.z);
    const float hi = x.axis == 0 ? h4.x : (x.axis == 1 ? h4.y : h4.z);
    const float c = __fmul_rn(0.5f, __fadd_rn(lo, hi));
    return bin_of(c, x.cbl[x.axis], x.scale[x.axis], kBins) <= static_cast<int>(x.bin);
}

// words[w] = ballot of "position goes to the left child" over positions 32w .. 32w+31 (0 outside splitting nodes)
__global__ void __launch_bounds__(256) kb_flags(Arrays A, uint32_t level, int parity) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    bool left = false;
    if (p < A.n) {
        const NodeAux &x = A.aux[A.node_of[parity][p]];
        if (x.level == level) left = goes_left(A, x, p, A.idx[parity][p]);
    }
    const uint32_t w = __ballot_sync(0xFFFFFFFFu, left);
    if ((threadIdx.x & 31) == 0 && p < A.n) A.words[p >> 5] = w;
}

// wscan[w] = sum of popc(words[0 .. w-1]); one block; total[0] = the grand total (may be null); zero[0] = 0 (may be
// null: the big phase clears the node list it has just consumed here, between two kb_split launches)
__global__ void __launch_bounds__(1024) kb_scan(const uint32_t *words, uint32_t *wscan, uint32_t n_words, uint32_t *total, uint32_t *zero) {
    __shared__ uint32_t part[1024];
    const uint32_t t = threadIdx.x;
    const uint32_t per = (n_words + 1023u) / 1024u;
    const uint32_t b = min(n_words, t * per), e = min(n_words, b + per);
    uint32_t s = 0;
    for (uint32_t i = b; i < e; ++i) s += __popc(words[i]);
    part[t] = s;
    __syncthreads();
    for (uint32_t off = 1; off < 1024; off <<= 1) {  // inclusive Hillis-Steele scan of the 1024 partial sums
        const uint32_t v = t >= off ? part[t - off] : 0u;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    uint32_t run = part[t] - s;
    for (uint32_t i = b; i < e; ++i) {
        wscan[i] = run;
        run += __popc(words[i]);
    }
    if (total && t == 1023) *total = part[1023];
    if (zero && t == 0) *zero = 0;
}

__device__ __forceinline__ uint32_t flags_before(const Arrays &A, uint32_t p) {
    return A.wscan[p >> 5] + __popc(A.words[p >> 5] & ((1u << (p & 31u)) - 1u));
}

__global__ void __launch_bounds__(256) kb_scatter(Arrays A, uint32_t level, int parity) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.n) return;
    const uint32_t slot = A.node_of[parity][p];
    const uint32_t prim = A.idx[parity][p];
    const NodeAux &x = A.aux[slot];
    uint32_t dst = p, to = slot;
    if (x.level == level) {
        const bool left = (A.words[p >> 5] >> (p & 31u)) & 1u;
        const uint32_t lefts = flags_before(A, p) - flags_before(A, x.begin);  // left-going positions of this node before p
        if (left) {
            dst = x.begin + lefts;
            to = slot + 1;
        } else {
            dst = x.begin + x.nleft + (p - x.begin - lefts);
            to = slot + 2 * x.nleft;
        }
    }
    A.idx[parity ^ 1][dst] = prim;
    A.node_of[parity ^ 1][dst] = to;
}

// ---- small phase: one warp per node of <= kSmall triangles, whole sub-tree ----------------------------------------------
struct SmallPrim {
    float lo[3], hi[3];
    uint32_t id;
};

__global__ void __launch_bounds__(128) kb_small(Arrays A, int parity) {
    __shared__ SmallPrim s_prims[4][kSmall];
    __shared__ uint32_t s_stack[4][kSmall + 2][3];
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31u, wib = threadIdx.x >> 5;
    const uint32_t w = blockIdx.x * 4 + wib;
    if (w >= A.c->n_small) return;
    const uint32_t root_slot = A.small[w];
    const uint32_t base = A.aux[root_slot].begin, n0 = A.aux[root_slot].count;
    SmallPrim *P = s_prims[wib];
    uint32_t *idx = A.idx[parity];
    if (lane < n0) {
        const uint32_t prim = idx[base + lane];
        const float4 l4 = A.plo[prim], h4 = A.phi[prim];
        P[lane] = SmallPrim{{l4.x, l4.y, l4.z}, {h4.x, h4.y, h4.z}, prim};
    }
    __syncwarp();
    int sp = 0;
    uint32_t(*S)[3] = s_stack[wib];
    if (lane == 0) {
        S[0][0] = root_slot;
        S[0][1] = 0;   // first triangle, relative to base
        S[0][2] = n0 | (A.aux[root_slot].depth << 8);
    }
    sp = 1;
    uint32_t max_depth = 0;
    while (sp > 0) {
        __syncwarp();
        --sp;
        const uint32_t slot = S[sp][0], b = S[sp][1], c = S[sp][2] & 255u, depth = S[sp][2] >> 8;
        __syncwarp();
        max_depth = depth > max_depth ? depth : max_depth;
        // this lane's triangle of the range, the node's box and centroid box
        SmallPrim me;
        float cen[3];
        float v[12];
        if (lane < c) {
            me = P[b + lane];
            for (int k = 0; k < 3; ++k) {
                cen[k] = __fmul_rn(0.5f, __fadd_rn(me.lo[k], me.hi[k]));
                v[k] = me.lo[k];
                v[3 + k] = me.hi[k];
                v[6 + k] = cen[k];
                v[9 + k] = cen[k];
            }
        } else {
            for (int k = 0; k < 3; ++k) {
                cen[k] = 0.0f;
                v[k] = v[6 + k] = HUGE_VALF;
                v[3 + k] = v[9 + k] = -HUGE_VALF;
            }
            me.id = 0;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1)
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const float o = __shfl_xor_sync(FULL, v[k], off);
                v[k] = (k % 6) < 3 ? fminf(v[k], o) : fmaxf(v[k], o);
            }
        Box box;
        for (int k = 0; k < 3; ++k) {
            box.lo[k] = v[k];
            box.hi[k] = v[3 + k];
        }
        rt_bvh_node &nd = A.nodes[slot];
        if (lane == 0) {
            for (int k = 0; k < 3; ++k) {
                nd.bmin[k] = box.lo[k];
                nd.bmax[k] = box.hi[k];
            }
        }
        auto make_leaf = [&]() {
            if (lane == 0) {
                nd.left_child = nd.right_child = RT_NO_CHILD;
                nd.obj_begin = base + b;
                nd.obj_end = base + b + c;
                A.last[base + b + c - 1] = 1;
            }
        };
        if (c <= 1) {
            make_leaf();
            continue;
        }
        float scale[3], cmin[3];
        for (int k = 0; k < 3; ++k) {
            const float ext = __fsub_rn(v[9 + k], v[6 + k]);
            cmin[k] = v[6 + k];
            scale[k] = ext > 0.0f ? __fdiv_rn(static_cast<float>(kSmallBins), ext) : 0.0f;
        }
        const bool force = static_cast<int>(depth) + ceil_log2(c) + 2 >= RT_STACK_SIZE - 2;
        // one candidate (axis, split after bin) per lane: 3 x 7 = 21 lanes, each sweeps the c triangles in shared memory
        float cost = HUGE_VALF;
        uint32_t cand_left = 0;
        const int axis = lane < 3 * (kSmallBins - 1) ? lane / (kSmallBins - 1) : 0, split = lane % (kSmallBins - 1);
        if (lane < 3 * (kSmallBins - 1) && !force && scale[axis] > 0.0f) {
            Box l, r;
            l.reset();
            r.reset();
            uint32_t cl = 0;
            for (uint32_t q = 0; q < c; ++q) {
                const SmallPrim &t = P[b + q];
                const float cc = __fmul_rn(0.5f, __fadd_rn(t.lo[axis], t.hi[axis]));
                if (bin_of(cc, cmin[axis], scale[axis], kSmallBins) <= split) {
                    l.grow(t.lo, t.hi);
                    ++cl;
                } else {
                    r.grow(t.lo, t.hi);
                }
            }
            if (cl > 0 && cl < c) {
                cost = __fadd_rn(__fmul_rn(static_cast<float>(cl), l.area()), __fmul_rn(static_cast<float>(c - cl), r.area()));
                cand_left = cl;
            }
        }
        // first minimum in (axis, bin) order, like the serial sweep of sah_build.h
        float best = cost;
        uint32_t best_lane = lane;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float oc = __shfl_xor_sync(FULL, best, off);
            const uint32_t ol = __shfl_xor_sync(FULL, best_lane, off);
            if (oc < best || (oc == best && ol < best_lane)) {
                best = oc;
                best_lane = ol;
            }
        }
        const bool have = best < HUGE_VALF;
        const float node_area = box.area();
        const float leaf_cost = __fmul_rn(static_cast<float>(c), node_area);
        bool left;
        uint32_t nleft;
        if (have && (c > kMaxLeaf || __fadd_rn(__fmul_rn(kTraversalCost, node_area), best) < leaf_cost)) {
            const int ba = best_lane / (kSmallBins - 1), bs = best_lane % (kSmallBins - 1);
            nleft = __shfl_sync(FULL, cand_left, best_lane);
            left = lane < c && bin_of(cen[ba], cmin[ba], scale[ba], kSmallBins) <= bs;
        } else if (c <= kMaxLeaf) {
            make_leaf();
            continue;
        } else {  // more than kMaxLeaf triangles that binning cannot separate: split by position
            nleft = c / 2;
            left = lane < nleft;
        }
        // stable partition inside the warp
        const uint32_t m_left = __ballot_sync(FULL, left);
        const uint32_t lt = (1u << lane) - 1u;
        const uint32_t m_valid = c >= 32 ? FULL : ((1u << c) - 1u);
        const uint32_t dst = left ? __popc(m_left & lt) : nleft + __popc(~m_left & m_valid & lt);
        __syncwarp();
        if (lane < c) P[b + dst] = me;
        if (lane == 0) {
            nd.left_child = slot + 1;
            nd.right_child = slot + 2 * nleft;
            nd.obj_begin = nd.obj_end = 0;
            S[sp][0] = slot + 2 * nleft;
            S[sp][1] = b + nleft;
            S[sp][2] = (c - nleft) | ((depth + 1) << 8);
            S[sp + 1][0] = slot + 1;
            S[sp + 1][1] = b;
            S[sp + 1][2] = nleft | ((depth + 1) << 8);
        }
        sp += 2;
    }
    __syncwarp();
    if (lane < n0) idx[base + lane] = P[lane].id;
    if (lane == 0) atomicMax(&A.c->max_depth, max_depth);
}

// ---- device layout of the triangles --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kb_tris(Arrays A, int parity, int with_tangents) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > A.n) return;
    if (k == A.n) {  // the null triangle: absent children of a wide node point here; pair loads may read one past a leaf
        DTri t;
        memset(&t, 0, sizeof t);
        t.id_last = RT_LAST_BIT;
        A.tris[k] = t;
        return;
    }
    const uint32_t id = A.idx[parity][k];
    const float *p = A.tri_pos + static_cast<size_t>(id) * 9;
    DTri t;
    t.ax = p[0]; t.ay = p[1]; t.az = p[2];
    t.e1x = __fsub_rn(p[3], p[0]); t.e1y = __fsub_rn(p[4], p[1]); t.e1z = __fsub_rn(p[5], p[2]);
    t.e2x = __fsub_rn(p[6], p[0]); t.e2y = __fsub_rn(p[7], p[1]); t.e2z = __fsub_rn(p[8], p[2]);
    t.pad0 = t.pad1 = 0.0f;
    t.pad2[0] = t.pad2[1] = t.pad2[2] = t.pad2[3] = 0.0f;
    t.id_last = id | (A.last[k] ? RT_LAST_BIT : 0u);
    A.tris[k] = t;
    const float *nn = A.tri_normals + static_cast<size_t>(id) * 9;
    const float *uv = A.tri_uv + static_cast<size_t>(id) * 6;
    DAttr a;
    a.n0x = nn[0]; a.n0y = nn[1]; a.n0z = nn[2];
    a.n1x = nn[3]; a.n1y = nn[4]; a.n1z = nn[5];
    a.n2x = nn[6]; a.n2y = nn[7]; a.n2z = nn[8];
    a.uv0x = uv[0]; a.uv0y = uv[1]; a.uv1x = uv[2]; a.uv1y = uv[3]; a.uv2x = uv[4]; a.uv2y = uv[5];
    a.material = A.tri_material[id];
    A.attrs[k] = a;
    if (with_tangents) {
        const float *tg = A.tri_tangents + static_cast<size_t>(id) * 9;
        DTangent d;
        d.t0x = tg[0]; d.t0y = tg[1]; d.t0z = tg[2];
        d.t1x = tg[3]; d.t1y = tg[4]; d.t1z = tg[5];
        d.t2x = tg[6]; d.t2y = tg[7]; d.t2z = tg[8];
        d.pad0 = d.pad1 = d.pad2 = 0.0f;
        A.tangents[k] = d;
    }
}

// ---- 4-wide collapse -----------------------------------------------------------------------------------------------------
struct Child {
    int32_t link;  // >= 0: binary inner node slot; < 0: ~first triangle of a leaf
    float lo[3], hi[3];
};
struct Opened {
    Child ch[4];
    int n;
};
__device__ __forceinline__ float child_area(const Child &c) {  // repack.h box_area(Child4)
    const float dx = c.hi[0] - c.lo[0], dy = c.hi[1] - c.lo[1], dz = c.hi[2] - c.lo[2];
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dy), __fmul_rn(dy, dz)), __fmul_rn(dz, dx));
}
__device__ __forceinline__ Child child_of(const rt_bvh_node *nodes, uint32_t i) {
    const rt_bvh_node &nd = nodes[i];
    Child c;
    c.link = (nd.left_child == RT_NO_CHILD && nd.right_child == RT_NO_CHILD) ? ~static_cast<int32_t>(nd.obj_begin) : static_cast<int32_t>(i);
    for (int k = 0; k < 3; ++k) {
        c.lo[k] = nd.bmin[k];
        c.hi[k] = nd.bmax[k];
    }
    return c;
}
// the 2..4 children of the wide node rooted at binary inner node `bin`: the inner child with the largest box is opened
// first (repack.h Built4::open)
__device__ Opened open_wide(const rt_bvh_node *nodes, uint32_t bin) {
    Opened o;
    o.n = 2;
    o.ch[0] = child_of(nodes, nodes[bin].left_child);
    o.ch[1] = child_of(nodes, nodes[bin].right_child);
    while (o.n < 4) {
        int best = -1;
        float best_area = -1.0f;
        for (int i = 0; i < o.n; ++i)
            if (o.ch[i].link >= 0) {
                const float a = child_area(o.ch[i]);
                if (a > best_area) {
                    best_area = a;
                    best = i;
                }
            }
        if (best < 0) break;
        const rt_bvh_node &nd = nodes[o.ch[best].link];
        o.ch[best] = child_of(nodes, nd.left_child);
        o.ch[o.n++] = child_of(nodes, nd.right_child);
    }
    return o;
}

__global__ void kb_mark_root(Arrays A) {
    const rt_bvh_node &r = A.nodes[0];
    if (r.left_child == RT_NO_CHILD && r.right_child == RT_NO_CHILD) return;  // the whole tree is one leaf
    A.mark[0] = 1;
    A.need[0] = 0;
    A.frontier[0][0] = 0;
    A.c->frontier[0] = 1;
}

// collapse level l: the wide roots in list l % 3 open their children; inner children are the wide roots of level l + 1
// (list (l + 1) % 3); the list of level l - 1, consumed by the previous launch, is emptied for level l + 2
__global__ void __launch_bounds__(128) kb_mark(Arrays A, uint32_t l) {
    const uint32_t cur = l % 3u, nxt = (l + 1u) % 3u;
    if (blockIdx.x == 0 && threadIdx.x == 0) A.c->frontier[(l + 2u) % 3u] = 0;
    const uint32_t n_f = A.c->frontier[cur];
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_f; k += gridDim.x * blockDim.x) {
        const uint32_t bin = A.frontier[cur][k];
        const Opened o = open_wide(A.nodes, bin);
        const uint32_t below = A.need[bin] + static_cast<uint32_t>(o.n - 1);
        atomicMax(&A.c->stack_need, below);
        for (int i = 0; i < o.n; ++i)
            if (o.ch[i].link >= 0) {
                A.mark[o.ch[i].link] = 1;
                A.need[o.ch[i].link] = below;
                A.frontier[nxt][atomicAdd(&A.c->frontier[nxt], 1u)] = static_cast<uint32_t>(o.ch[i].link);
            }
    }
}

__global__ void __launch_bounds__(256) kb_markwords(Arrays A, uint32_t n_slots) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    const bool m = s < n_slots && A.mark[s];
    const uint32_t w = __ballot_sync(0xFFFFFFFFu, m);
    if ((threadIdx.x & 31) == 0 && s < n_slots) A.words[s >> 5] = w;
}

__global__ void __launch_bounds__(128) kb_emit(Arrays A, uint32_t n_slots) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_slots || !A.mark[s]) return;
    const Opened o = open_wide(A.nodes, s);
    QNode4 q;
    memset(&q, 0, sizeof q);
    const int32_t null_leaf = ~static_cast<int32_t>(A.n);
    for (int i = 0; i < 4; ++i) {
        if (i >= o.n) q.link[i] = null_leaf;
        else if (o.ch[i].link < 0) q.link[i] = o.ch[i].link;
        else q.link[i] = static_cast<int32_t>(flags_before(A, static_cast<uint32_t>(o.ch[i].link)));
    }
    for (int a = 0; a < 3; ++a) {
        float lo[4], hi[4];
        uint8_t ql[4] = {255, 255, 255, 255}, qh[4] = {0, 0, 0, 0};  // absent child: inverted box
        for (int i = 0; i < o.n; ++i) {
            lo[i] = o.ch[i].lo[a];
            hi[i] = o.ch[i].hi[a];
        }
        if (!rt::detail::quantize_axis_n(lo, hi, o.n, q.org[a], ql, qh)) atomicOr(&A.c->error, 1u);
        q.lo[a] = static_cast<uint32_t>(ql[0]) | static_cast<uint32_t>(ql[1]) << 8 | static_cast<uint32_t>(ql[2]) << 16 | static_cast<uint32_t>(ql[3]) << 24;
        q.hi[a] = static_cast<uint32_t>(qh[0]) | static_cast<uint32_t>(qh[1]) << 8 | static_cast<uint32_t>(qh[2]) << 16 | static_cast<uint32_t>(qh[3]) << 24;
    }
    A.qnodes4[flags_before(A, s)] = q;
}

// ---- refit (rt_gpu_update_geometry) ------------------------------------------------------------------------------------
// The tree keeps its topology: the binary slots, the triangle order idx[parity], the leaf ends `last` and the 4-wide
// grouping.  Only boxes change.  State recorded at the first update after an upload, from the pristine tree:
//   kr_levels_init / kr_levels   the used binary slots, level by level from the root (unused slots hold undefined data)
//   kr_wide_slots                for each 4-wide node, the binary slot behind each child (open_wide picks children by
//                                box area, so collapsing the refit boxes again could regroup)
// Every update then runs kr_refit once per binary level from the deepest up, kr_requant over the 4-wide nodes, and kb_tris.
// Boxes reduce with fminf / fmaxf, as kb_setup, kb_split and kb_small do, so refitting to the uploaded positions
// reproduces the uploaded tree bit for bit.
constexpr uint32_t kMaxLevels = RT_STACK_SIZE + 2;

struct Refit {
    uint32_t *order;   // [n_slots] used binary slots, level by level
    uint32_t *lstart;  // [kMaxLevels] first entry of each level in `order`
    uint32_t *lcount;  // [kMaxLevels] entries of each level
    int32_t *wslot;    // [4 * n_wide] binary slot behind child i of 4-wide node w; -1: absent child
};

__global__ void kr_levels_init(Refit R) {
    R.lstart[0] = 0;
    R.lcount[0] = 1;
    R.order[0] = 0;
}

// level l lists its inner nodes' children as level l + 1 (appended right behind level l)
__global__ void __launch_bounds__(256) kr_levels(Arrays A, Refit R, uint32_t l) {
    const uint32_t begin = R.lstart[l], cnt = R.lcount[l], next = begin + cnt;
    if (blockIdx.x == 0 && threadIdx.x == 0) R.lstart[l + 1] = next;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < cnt; k += gridDim.x * blockDim.x) {
        const rt_bvh_node &nd = A.nodes[R.order[begin + k]];
        if (nd.left_child == RT_NO_CHILD) continue;
        const uint32_t at = next + atomicAdd(&R.lcount[l + 1], 2u);
        R.order[at] = nd.left_child;
        R.order[at + 1] = nd.right_child;
    }
}

// open_wide, keeping the binary slot of every child; the links it implies are checked against kb_emit's (error bit 1)
__global__ void __launch_bounds__(128) kr_wide_slots(Arrays A, Refit R, uint32_t n_slots) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_slots || !A.mark[s]) return;
    const rt_bvh_node *nodes = A.nodes;
    uint32_t slot[4] = {nodes[s].left_child, nodes[s].right_child, 0, 0};
    int n = 2;
    auto inner = [&](uint32_t i) { return nodes[i].left_child != RT_NO_CHILD || nodes[i].right_child != RT_NO_CHILD; };
    while (n < 4) {
        int best = -1;
        float best_area = -1.0f;
        for (int i = 0; i < n; ++i)
            if (inner(slot[i])) {
                const float a = child_area(child_of(nodes, slot[i]));
                if (a > best_area) {
                    best_area = a;
                    best = i;
                }
            }
        if (best < 0) break;
        const uint32_t b = slot[best];
        slot[best] = nodes[b].left_child;
        slot[n++] = nodes[b].right_child;
    }
    const uint32_t w = flags_before(A, s);
    const QNode4 &q = A.qnodes4[w];
    bool same = true;
    for (int i = 0; i < 4; ++i) {
        int32_t link = ~static_cast<int32_t>(A.n);
        if (i < n) link = inner(slot[i]) ? static_cast<int32_t>(flags_before(A, slot[i])) : ~static_cast<int32_t>(nodes[slot[i]].obj_begin);
        same = same && link == q.link[i];
        R.wslot[4 * w + i] = i < n ? static_cast<int32_t>(slot[i]) : -1;
    }
    if (!same) atomicOr(&A.c->error, 2u);
}

// the binary nodes of one level: a leaf becomes the union of its triangles' boxes (kb_setup's), an inner node the union
// of its children's.  Non-finite vertices set error bit 0, as in kb_setup.
__global__ void __launch_bounds__(256) kr_refit(Arrays A, Refit R, uint32_t begin, uint32_t cnt, int parity) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= cnt) return;
    rt_bvh_node &nd = A.nodes[R.order[begin + k]];
    float lo[3] = {HUGE_VALF, HUGE_VALF, HUGE_VALF}, hi[3] = {-HUGE_VALF, -HUGE_VALF, -HUGE_VALF};
    if (nd.left_child == RT_NO_CHILD) {
        bool finite = true;
        for (uint32_t p = nd.obj_begin; p < nd.obj_end; ++p) {
            const float *v = A.tri_pos + static_cast<size_t>(A.idx[parity][p]) * 9;
            for (int d = 0; d < 3; ++d) {
                const float a = v[d], b = v[3 + d], c = v[6 + d];
                lo[d] = fminf(lo[d], fminf(a, fminf(b, c)));
                hi[d] = fmaxf(hi[d], fmaxf(a, fmaxf(b, c)));
                finite = finite && rt::detail::finite_f(a) && rt::detail::finite_f(b) && rt::detail::finite_f(c);
            }
        }
        if (!finite) atomicOr(&A.c->error, 1u);
    } else {
        const rt_bvh_node &l = A.nodes[nd.left_child], &r = A.nodes[nd.right_child];
        for (int d = 0; d < 3; ++d) {
            lo[d] = fminf(l.bmin[d], r.bmin[d]);
            hi[d] = fmaxf(l.bmax[d], r.bmax[d]);
        }
    }
    for (int d = 0; d < 3; ++d) {
        nd.bmin[d] = lo[d];
        nd.bmax[d] = hi[d];
    }
}

// kb_emit's quantisation of every 4-wide node from the refit binary boxes of its recorded children; links are kept
__global__ void __launch_bounds__(128) kr_requant(Arrays A, Refit R, uint32_t n_wide) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_wide) return;
    QNode4 q;
    memset(&q, 0, sizeof q);
    int n = 0;
    for (int i = 0; i < 4; ++i) {
        q.link[i] = A.qnodes4[w].link[i];
        n += R.wslot[4 * w + i] >= 0 ? 1 : 0;
    }
    for (int a = 0; a < 3; ++a) {
        float lo[4], hi[4];
        uint8_t ql[4] = {255, 255, 255, 255}, qh[4] = {0, 0, 0, 0};  // absent child: inverted box
        for (int i = 0; i < n; ++i) {
            const rt_bvh_node &c = A.nodes[R.wslot[4 * w + i]];
            lo[i] = c.bmin[a];
            hi[i] = c.bmax[a];
        }
        if (!rt::detail::quantize_axis_n(lo, hi, n, q.org[a], ql, qh)) atomicOr(&A.c->error, 1u);
        q.lo[a] = static_cast<uint32_t>(ql[0]) | static_cast<uint32_t>(ql[1]) << 8 | static_cast<uint32_t>(ql[2]) << 16 | static_cast<uint32_t>(ql[3]) << 24;
        q.hi[a] = static_cast<uint32_t>(qh[0]) | static_cast<uint32_t>(qh[1]) << 8 | static_cast<uint32_t>(qh[2]) << 16 | static_cast<uint32_t>(qh[3]) << 24;
    }
    A.qnodes4[w] = q;
}

}  // namespace rtb

#endif  // RT_GPU_BUILD_CUH
