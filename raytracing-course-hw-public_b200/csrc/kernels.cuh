// kernels.cuh — the wavefront kernels (sm_100a).  One "batch" = npix pixels x k samples = N paths:
//
//   k_generate   N paths: Philox pixel jitter -> camera ray (gen_ray, raytracer.h:527-538), 8 x 4 pixel tiles per warp
//   for bounce b in [0, ray_depth):
//     k_lightpdf_list  (b > 0, scenes with lights) all-hit traversal of the light BVH (bvh_mix_dist::pdf,
//                raytracer.h:363) for the pending rays of queue b that k_shade(b - 1) found inside the box of all lights
//     k_extend   closest-hit BVH traversal of queue b (cast_ray -> BVH::intersect_ray, bvh.h:170-235)
//     k_shade    resolve the previous bounce with that light pdf, hit data + shade() state transition
//                (raytracer.h:555-591), survivors compacted into queue b+1 with warp-aggregated
//                (__ballot/__popc) appends; light-box test of the rays it queues
//   k_accumulate per-sample NaN scrub + per-pixel float sums (render_pixel, raytracer.h:607-627)
// Small batches run k_extend / k_shade once per HALF of a queue, the halves on two streams (rt_gpu.cu, enqueue_render).
//
// Path state is SoA of float4 (128-bit coalesced loads/stores), ping-ponged between queue b and b+1:
//   q_o   = (origin.xyz,     pixel index bits)
//   q_d   = (direction.xyz,  sample index bits)
//   q_thr = (throughput.rgb [x f_cos when pending], p_partial >= 0 when the path's pdf still needs the light
//            pdf of this ray ("pending", also bit 31 of the sample index), else -1)
//   hit   = (t, beta, gamma, BVH-order triangle index bits or -1)      written by extend, read by shade
//   lpdf  = light pdf of the queued ray, one array per queue parity     written by shade (0: outside the light box) and
//           k_lightpdf_list for the pending rays of the queue, read by the next shade
//   llist = queue indices of the pending rays inside the light box      written by shade, read by k_lightpdf_list
//   rad   = per-path radiance accumulator, indexed by the path's fixed slot (no atomics: one owner)
// extend and shade are persistent: grid = SMs x resident CTAs, each warp pulls queue entries (128 / 32 at a time) from
// a device counter, so no host round trip is needed to size a launch.
#ifndef RT_KERNELS_CUH
#define RT_KERNELS_CUH

#include <cuda_runtime.h>

#include "pt_core.cuh"
#include "rt_types.h"

namespace rt {

struct BatchParams {
    uint32_t pix0;      // first pixel (row-major index) of this batch
    uint32_t npix;      // pixels in this batch
    uint32_t s0;        // first sample index of this batch
    uint32_t k;         // samples per pixel in this batch
    uint32_t width, height;
    uint32_t k0, k1;    // Philox key
    uint32_t centre;    // 1: pixel-centre rays without jitter (gen_ray(camera, x, y), raytracer.h:516-525)
    uint32_t tiled;     // 1: queue 0 holds the camera rays in 8 x 4 pixel tiles (one warp = one tile) instead of row-major
};

// The ping-pong parity is resolved on the HOST (in = queue b, out = queue b + 1): indexing pointer arrays of a kernel
// parameter with a run-time `bounce & 1` makes nvcc copy the whole parameter to local memory and re-load the
// pointers with LDL inside k_shade's loop (round 1: 37 % of its load requests).
struct Queues {
    const float4 *o_in, *d_in, *thr_in;  // queue b   (k_generate writes queue 0 through the *_out pointers)
    float4 *o_out, *d_out, *thr_out;     // queue b+1
    float4 *hit;
    float4 *rad;
    // Every counter sits in its own 256-byte line (index * kCounterStride).  Packed into one line (round 1), k_shade ran
    // 13 % slower whenever a small allocation preceded the queue arena (the "one process in six" / every NCCL rank
    // slow mode: 28.4 instead of 25.0 ms per 128 spp, reproducible with a 2 MB dummy cudaMalloc); padded, both
    // placements run at 25.0 (profiles/r2_bimodal.md).  Fewer atomics (128 entries per fetch, output slots reserved in
    // per-warp chunks) were measured as well and are slower (27.3: the extra loop level costs 8 registers).
    uint32_t *count;        // [ray_depth + 1] queue sizes
    uint32_t *fetch_ext;    // [ray_depth] work-fetch cursors of k_extend
    uint32_t *fetch_shade;  // [ray_depth] work-fetch cursors of k_shade
    unsigned long long *stats;  // [4] extension rays, light pdf rays, shades, samples
    float *lpdf;                // light pdf (bvh_mix_dist::pdf) of the pending rays of queue b: written by k_lightpdf_list
                                // (k_extend in the 8-wide build), read by k_shade
    float *lpdf_out;            // the same for queue b + 1.  k_shade stores the zeros of the rays that miss the light box
                                // there while other warps still read `lpdf` of queue b: two arrays, like the records
    uint32_t *light_list;       // RT_LIGHT_KERNEL == 2: indices (in the OUT queue) of the pending rays that pass the light box
    uint32_t *light_count;      // [ray_depth + 1] sizes of that list, per queue
};

// A launch of k_extend / k_shade handles the whole queue or one half of it: the host runs the two halves on two streams
// so that one half's kernels fill the SMs the other half's draining kernel leaves idle (rt_gpu.cu); each half has its
// own work-fetch cursors (fetch_ext / fetch_shade point at them).  The part travels in the high bits of the kernels'
// `bounce` argument (kPartFirst / kPartSecond): growing the Queues parameter by two words cost k_shade eight registers.
constexpr uint32_t kPartShift = 16, kPartFirst = 1u << kPartShift, kPartSecond = 2u << kPartShift;
// [part_begin, part_end) of the queue entries a launch handles; the halves meet at a multiple of 128 (k_extend's ray
// block).  The begin is a function of the end, so that the kernels need not keep it in a register.
__device__ __forceinline__ uint32_t part_end(uint32_t part, uint32_t count) {
    return part == kPartFirst ? (count >> 1) & ~127u : count;
}
__device__ __forceinline__ uint32_t part_begin(uint32_t part, uint32_t end) {  // end = part_end(part, count)
    return part == kPartSecond ? (end >> 1) & ~127u : 0u;
}

// Queue records are read once and written once per bounce (streaming), the scene is re-read by every ray: with
// RT_QUEUE_STREAMING the queue accesses carry the evict-first hint (ld/st.global.cs) so that they do not push nodes,
// triangles and attributes out of the L2.  Measured on the B200 (k_extend / k_shade ms per 128 spp): off 84.9 / 25.7,
// k_extend's accesses only 84.0 / 25.8 (the default), everything incl. the radiance sums 83.7 / 28.6.  An explicit L2
// persisting window over the scene arrays (cudaAccessPropertyPersisting) changed nothing and was removed.
#ifndef RT_QUEUE_STREAMING
#define RT_QUEUE_STREAMING 1
#endif
// bit 0: k_extend's ray loads and hit stores; bit 1: k_shade's record loads; bit 2: k_shade's / k_generate's record
// stores; bit 3: the radiance accumulator
template <int BIT> __device__ __forceinline__ float4 q_load(const float4 *p) { return (RT_QUEUE_STREAMING >> BIT) & 1 ? __ldcs(p) : *p; }
template <int BIT> __device__ __forceinline__ float q_load(const float *p) { return (RT_QUEUE_STREAMING >> BIT) & 1 ? __ldcs(p) : *p; }
template <int BIT> __device__ __forceinline__ void q_store(float4 *p, float4 v) {
    if ((RT_QUEUE_STREAMING >> BIT) & 1) __stcs(p, v);
    else *p = v;
}
template <int BIT> __device__ __forceinline__ void q_store(float *p, float v) {
    if ((RT_QUEUE_STREAMING >> BIT) & 1) __stcs(p, v);
    else *p = v;
}

#ifndef RT_EXT_THREADS
#define RT_EXT_THREADS 128  // threads per CTA of k_extend (and k_extend8)
#endif
constexpr int kExtendThreads = RT_EXT_THREADS;
constexpr int kShadeThreads = 128;
#ifndef RT_COUNTER_STRIDE
#define RT_COUNTER_STRIDE 64  // uint32 per counter slot (256 B); 1 = packed (round 1)
#endif
constexpr uint32_t kCounterStride = RT_COUNTER_STRIDE;

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// Position pl of a whole-image queue in 8 x 4 pixel tiles (one warp = one tile; width % 8 == 0, height % 4 == 0)
__device__ __forceinline__ uint32_t tiled_pixel(uint32_t pl, uint32_t width) {
    const uint32_t tile = pl >> 5, in = pl & 31u, tiles_x = width >> 3;
    const uint32_t ty = tile / tiles_x, tx = tile - ty * tiles_x;
    return (ty * 4u + (in >> 3)) * width + tx * 8u + (in & 7u);
}

// The queue-0 record of a camera ray (origin o, direction dir) of Philox key (pixel, sample) at queue position `slot`,
// its radiance slot `rad_slot` cleared
__device__ __forceinline__ void emit_ray_record(const BatchParams &bp, const Queues &q, uint32_t slot, uint32_t rad_slot, uint32_t pixel,
                                                uint32_t sample, f3 o, f3 dir) {
    q_store<2>(q.o_out + slot, make_float4(o.x, o.y, o.z, __uint_as_float(pixel)));
    q_store<2>(q.d_out + slot, make_float4(dir.x, dir.y, dir.z, __uint_as_float(sample)));
    q_store<2>(q.thr_out + slot, make_float4(1.0f, 1.0f, 1.0f, -1.0f));
    q_store<3>(q.rad + rad_slot, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
}

// The camera ray through pixel (px, py) of `cam` for Philox key (pixel, sample) into queue position `slot`, its radiance
// slot `rad_slot` cleared.  The multi-view k_generate_views (views.cuh) keys a view's pixel apart from its (px, py).
__device__ __forceinline__ void emit_camera_ray_at(const Camera &cam, const BatchParams &bp, const Queues &q, uint32_t slot, uint32_t rad_slot,
                                                   uint32_t pixel, uint32_t px, uint32_t py, uint32_t sample) {
    const RngKey key{pixel, sample, bp.k0, bp.k1};
    float jx = 0.5f, jy = 0.5f;
    if (!bp.centre) {
        const u4 r = rng_jitter(key);
        jx = u01(r.x);
        jy = u01(r.y);
    }
    const f3 dir = camera_dir(cam, static_cast<float>(px) + jx, static_cast<float>(py) + jy);
    emit_ray_record(bp, q, slot, rad_slot, pixel, sample, cam.pos, dir);
}

// The camera ray of row-major (pixel, sample).  k_generate and the adaptive k_generate_active (adaptive.cuh) both go
// through here.
__device__ __forceinline__ void emit_camera_ray(const Camera &cam, const BatchParams &bp, const Queues &q, uint32_t slot, uint32_t rad_slot,
                                                uint32_t pixel, uint32_t sample) {
    const uint32_t py = pixel / bp.width;
    const uint32_t px = pixel - py * bp.width;
    emit_camera_ray_at(cam, bp, q, slot, rad_slot, pixel, px, py, sample);
}

__global__ void __launch_bounds__(256) k_generate(Camera cam, BatchParams bp, Queues q) {
    const uint32_t n = bp.npix * bp.k;
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot == 0) {
        q.count[0] = n;
        atomicAdd(q.stats + 3, static_cast<unsigned long long>(n));
    }
    if (slot >= n) return;
    const uint32_t j = slot / bp.npix;
    const uint32_t pl = slot - j * bp.npix;
    // The order of queue 0 is free (a path's radiance slot follows from its pixel and sample, not from its queue
    // position): with one 8 x 4 tile per warp instead of a 32 x 1 strip the camera rays of a warp share more of their
    // traversal (bounce 0 is a quarter of k_extend's time).  Whole-image batches only (the host sets bp.tiled).  The
    // slots of the batch are a permutation of its queue positions, so clearing rad at `slot` clears all of them.
    const uint32_t pixel = bp.tiled ? tiled_pixel(pl, bp.width) : bp.pix0 + pl;
    emit_camera_ray(cam, bp, q, slot, slot, pixel, bp.s0 + j);
}

// one term of bvh_mix_dist::pdf: the light triangle `le` (normal, area) hit at distance t along d
// (raytracer.h:79-84,255-261: every hit counts, occluded or not, both faces); the 1 / n_lights is applied to the sum
__device__ __forceinline__ float light_pdf_term(f3 d, float t, f4 le) {
    const f3 xy = d * t;  // y - x
    const float d2 = len2(xy);
    const f3 w = xy * rsqrtf(d2);
    return __fdividef(d2, fabsf(dot(w, mk3(le.x, le.y, le.z))) * le.w);  // MUFU.RCP: 2e-7 of a pdf term
}

// ---- k_extend -----------------------------------------------------------------------------------------
// Closest-hit traversal over the 4-wide quantised nodes (QNode4), warp-synchronous "while-while" with one postponed
// leaf per lane (Aila & Laine 2009 style speculative traversal) and per-lane ray refill:
//   * every loop condition is a warp vote (__any_sync / __ballot_sync), so the 32 lanes re-converge at
//     each phase boundary instead of drifting apart (the naive per-thread loop ran its triangle tests
//     with 2 of 32 lanes active);
//   * inner phase: one iteration = at most one stack pop, then at most one node step per lane, then the leaf
//     check, all predicated (no per-lane loops: the pop-until-useful loop of the first version ran with 2 of 32
//     lanes active and was 9 % of the kernel's instructions).  The first leaf a lane meets is postponed and the
//     lane keeps descending speculatively; a lane that meets a second leaf waits.  The phase ends when fewer
//     than kMinSearching lanes are still looking for their first leaf;
//   * leaf phase: all postponed leaves are intersected together, two triangles per iteration;
//   * a lane whose ray is finished stores its hit and takes the next ray from a warp-local block of
//     kRayBlock queue entries (one atomicAdd per block), ranks handed out with __ballot_sync/__popc.
// Visiting order (near child first, ties left first, bvh.h:216) and strictly-closer-wins (bvh.h:132)
// are those of closest_hit_q4() in pt_core.cuh, so both give the same hit.
//
// With RT_LIGHT_KERNEL == 0 (the 8-wide build's setting; the default until r2_v4) a pending ray (bit 31 of its sample
// index) is traversed twice: first through the light BVH, all hits, summing bvh_mix_dist::pdf (raytracer.h:363-375;
// best_t stays +inf, so nothing is culled), then through the scene BVH for the closest hit, both in the same
// warp-synchronous loops.  By default the light query runs in k_lightpdf_list and this kernel sees scene rays only.
//
// Compile-time knobs (A/B-tested on the B200, DESIGN.md "k_extend"; defaults = the fastest measured).  Alternatives
// that were measured and removed from the source: 2-wide 32-byte nodes, 64-byte full-precision nodes, node step before
// the pop, two pops per step, one triangle per leaf iteration, light-to-scene switch in the refill section.
#ifndef RT_EXT_SMEM_STACK
#define RT_EXT_SMEM_STACK 16  // traversal-stack entries per thread kept in shared memory (0: all in local memory)
#endif
#ifndef RT_EXT_MIN_SEARCH
#define RT_EXT_MIN_SEARCH 20  // leave the inner phase when fewer lanes than this still look for their first leaf
#endif
#ifndef RT_EXT_STEPS_PER_VOTE
#define RT_EXT_STEPS_PER_VOTE 3  // 1 / 2 / 3 / 4 -> 103.4 / 100.4 / 99.3 / 100.4 ms of k_extend per 128 spp
#endif
#ifndef RT_EXT_MINB
#define RT_EXT_MINB 9  // minimum resident CTAs per SM asked of the compiler: 9 = 56 registers, no spills since the light traversal left the kernel (8: +0.6 %, 10: spills, +6 %)
#endif
constexpr int32_t kLinkDone = static_cast<int32_t>(0x80000000u);  // nothing left to traverse
constexpr int32_t kLinkPop = static_cast<int32_t>(0x80000001u);   // take the next entry from the stack
constexpr uint32_t kRayBlock = 128;
// Traversal stack: the first kSmemStack entries of every thread live in shared memory ([entry][thread], so
// a warp's access is bank-conflict free whatever the lanes' stack pointers are); deeper entries (rare: the
// ordered traversal seldom holds more than a dozen postponed children) overflow to local memory.  The
// all-local stack cost one 32 B sector of L1 data-pipe time per lane and push (write-through to L2: 4.2 GB
// per launch, 31 % of the kernel's L1 sectors — profiles/r1_v2_k_extend_ncu_full.csv).
constexpr int kSmemStack = RT_EXT_SMEM_STACK;
constexpr int kMinSearching = RT_EXT_MIN_SEARCH;
constexpr int kStepsPerVote = RT_EXT_STEPS_PER_VOTE;
constexpr uint32_t kNoRay = 0xFFFFFFFFu;

// MUFU.RCP (1 ulp): one instruction instead of the IEEE division's Newton step + slow path
__device__ __forceinline__ float rcp_rn(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// L1 eviction hints of k_extend's scene fetches: 0 none, 1 no_allocate, 2 evict_last, 3 evict_first.  Triangles are
// read about once per ray and from a 16 MB array; nodes are re-read (the top of the tree by every ray).
#ifndef RT_EXT_NODE_L1
#define RT_EXT_NODE_L1 0  // no_allocate on the nodes: +9 % (an L1 hit costs 0.7 data-pipe cycles per lane, a miss 1.0); evict_last: +1 %
#endif
#ifndef RT_EXT_TRI_L1
#define RT_EXT_TRI_L1 1  // no_allocate: k_extend 159.5 -> 157.3 ms per 256 spp (evict_first: no change; evict_last on the nodes: +1 %)
#endif
// bvh_mix_dist::pdf of the pending rays: 0 = a traversal mode of k_extend (rounds 1 / 2, and the 8-wide build);
// 2 = k_shade tests the ray it queues against the box of all lights and lists those that pass, k_lightpdf_list
// traverses the light BVH for them (1, a light kernel that scanned the whole queue, was measured and removed)
#ifndef RT_LIGHT_KERNEL
#define RT_LIGHT_KERNEL 2
#endif
#if defined(RT_EXT_WIDE8) && RT_EXT_WIDE8
#undef RT_LIGHT_KERNEL
#define RT_LIGHT_KERNEL 0
#endif
#ifndef RT_EXT_SPLIT_NODES
#define RT_EXT_SPLIT_NODES 1  // node halves from two arrays of 32-byte stride (DBvh::q4lo) instead of 64-byte records
#endif
template <int H> __device__ __forceinline__ f8 ld8h(const void *p) {
    f8 v;
    if (H == 1)
        asm("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
            : "=f"(v.a), "=f"(v.b), "=f"(v.c), "=f"(v.d), "=f"(v.e), "=f"(v.f), "=f"(v.g), "=f"(v.h) : "l"(p));
    else if (H == 2)
        asm("ld.global.nc.L1::evict_last.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
            : "=f"(v.a), "=f"(v.b), "=f"(v.c), "=f"(v.d), "=f"(v.e), "=f"(v.f), "=f"(v.g), "=f"(v.h) : "l"(p));
    else if (H == 3)
        asm("ld.global.nc.L1::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
            : "=f"(v.a), "=f"(v.b), "=f"(v.c), "=f"(v.d), "=f"(v.e), "=f"(v.f), "=f"(v.g), "=f"(v.h) : "l"(p));
    else
        v = ld8(p);
    return v;
}
template <int H> __device__ __forceinline__ f4 ld4h(const void *p) {
    f4 v;
    if (H == 1)
        asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    else if (H == 2)
        asm("ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    else if (H == 3)
        asm("ld.global.nc.L1::evict_first.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    else
        v = ld4(p);
    return v;
}

__device__ __forceinline__ bool link_is_leaf(int32_t link) { return link < 0 && link != kLinkDone && link != kLinkPop; }

__global__ void __launch_bounds__(kExtendThreads, RT_EXT_MINB)
    k_extend(DBvh bvh, DBvh lbvh, const DLight *__restrict__ light_extra, float inv_n_lights, float eps, Queues q, uint32_t bounce_part,
             uint32_t one) {
    // `one` = 0x3F800000, passed as an argument so that it is not an immediate (see qplane() in pt_core.cuh)
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t part = bounce_part & ~(kPartFirst - 1u), bounce = bounce_part & (kPartFirst - 1u);
    const uint32_t count = part_end(part, q.count[bounce * kCounterStride]);  // this launch's part of the queue: [part_begin, count)
    const float4 *__restrict__ qo = q.o_in;
    const float4 *__restrict__ qd = q.d_in;
    uint32_t *cursor = q.fetch_ext + bounce * kCounterStride;
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;

    // postponed far children: (link, entry distance) pairs, [entry][thread]: one 64-bit shared-memory access per entry
    // (two 32-bit planes cost the same L1 wavefronts but twice the instructions: +1.4 % kernel time)
    __shared__ uint2 s_stack[(kSmemStack > 0 ? kSmemStack : 1) * kExtendThreads];
#define RT_ST(p, l, t) (p)[0] = make_uint2(static_cast<uint32_t>(l), __float_as_uint(t))
#define RT_LD(p, l, t)                   \
    do {                                 \
        const uint2 e_ = (p)[0];         \
        l = static_cast<int32_t>(e_.x);  \
        t = __uint_as_float(e_.y);       \
    } while (0)
    // the deeper part of the stack; the upload path guarantees that no ray needs more than RT_EXT_STACK_CAP entries
    // (PackedBvh::stack_need4, checked in pack_bvh), so push() carries no bounds check
    float2 overflow[RT_EXT_STACK_CAP - kSmemStack];
    uint2 *top = s_stack + threadIdx.x;  // slot of the NEXT push (valid while sp < kSmemStack)
    int sp = 0;
    int32_t link = kLinkDone;  // >= 0 inner node, kLinkPop / kLinkDone, otherwise a leaf (~first triangle)
    int32_t leaf = 0;          // postponed leaf link (always < 0) or 0 = none
    uint32_t ray = kNoRay;     // queue index; bit 31: pending (its light pdf is wanted)
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 1), idir = mk3(0, 0, 1);
    float best_t = INFINITY, best_b = 0.0f, best_c = 0.0f;
    int32_t best_tri = -1;
#if RT_LIGHT_KERNEL
    constexpr bool leaf_l = false;  // the light BVH is traversed by k_lightpdf
#else
    bool lmode = false;   // the lane is in the light BVH
    bool leaf_l = false;  // the postponed leaf belongs to the light BVH
    float lsum = 0.0f;
#endif
    const int32_t scene_root = bvh.root4 == RT_LINK_NONE ? kLinkDone : bvh.root4;
#if RT_EXT_SPLIT_NODES
    const char *node_base = bvh.q4lo;
    const size_t hi_off = bvh.q4_hi_off;
#else
    const QNode4 *node_base = bvh.qnodes4;
#endif
    uint32_t pool_next = 0, pool_end = 0;  // warp-uniform block of queue entries
    bool exhausted = false;                 // warp-uniform

    for (;;) {
        // ---- retire finished rays, refill idle lanes ---------------------------------------------------
        const bool idle = link == kLinkDone && leaf == 0;
        if (idle && ray != kNoRay) {
            const uint32_t r = ray & 0x7FFFFFFFu;
#if !RT_LIGHT_KERNEL
            if (ray >> 31) q_store<0>(q.lpdf + r, lsum * inv_n_lights);  // 0 when the scene has no light BVH
#endif
            q_store<0>(q.hit + r, make_float4(best_t, best_b, best_c, __int_as_float(best_tri)));
            ray = kNoRay;
        }
        const uint32_t m_idle = __ballot_sync(FULL, idle);
        if (m_idle) {
            if (pool_next == pool_end && !exhausted) {  // one atomicAdd per kRayBlock rays
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(cursor, kRayBlock);
                base = __shfl_sync(FULL, base, 0) + part_begin(part, count);
                if (base >= count) {
                    exhausted = true;
                } else {
                    pool_next = base;
                    pool_end = base + kRayBlock < count ? base + kRayBlock : count;
                }
            }
            const uint32_t avail = pool_end - pool_next;
            const uint32_t n_idle = static_cast<uint32_t>(__popc(m_idle));
            const uint32_t take = n_idle < avail ? n_idle : avail;
            const uint32_t rank = static_cast<uint32_t>(__popc(m_idle & lt_mask));
            if (idle && rank < take) {
                ray = pool_next + rank;
                const float4 o4 = q_load<0>(qo + ray), d4 = q_load<0>(qd + ray);
                o = mk3(o4.x, o4.y, o4.z);
                d = mk3(d4.x, d4.y, d4.z);
                idir = mk3(rcp_rn(d.x), rcp_rn(d.y), rcp_rn(d.z));
                best_t = INFINITY;
                best_b = best_c = 0.0f;
                best_tri = -1;
                sp = 0;
                top = s_stack + threadIdx.x;
#if RT_LIGHT_KERNEL
                link = scene_root;  // a leaf root is postponed in the first step
#else
                lsum = 0.0f;
                lmode = (__float_as_uint(d4.w) >> 31) != 0u && lbvh.root4 != RT_LINK_NONE;
                ray |= __float_as_uint(d4.w) & 0x80000000u;
#if RT_EXT_SPLIT_NODES
                node_base = lmode ? lbvh.q4lo : bvh.q4lo;
#else
                node_base = lmode ? lbvh.qnodes4 : bvh.qnodes4;
#endif
                link = lmode ? lbvh.root4 : scene_root;  // a leaf root is postponed in the first step
#endif
            }
            pool_next += take;
            if (avail == 0 && m_idle == FULL) break;  // queue drained and nothing in flight
        }
        const bool can_refill = !exhausted || pool_next != pool_end;  // warp-uniform

        // ---- inner phase -------------------------------------------------------------------------------
        for (;;) {
            // phase vote, once per kStepsPerVote steps: go on while at least kMinSearching lanes still look
            // for their first leaf (a lane that has nothing to do in a step simply idles through it)
            const uint32_t m_search = __ballot_sync(FULL, leaf == 0 && link != kLinkDone);
            if (__popc(m_search) < kMinSearching) {
                if (m_search == 0) break;
                // few lanes still search: go and do useful work for the others if there is any (pending
                // leaves to intersect, or finished lanes that can take a new ray); else keep going
                if (__any_sync(FULL, leaf != 0 || (can_refill && link == kLinkDone))) break;
            }
#pragma unroll
            for (int step = 0; step < kStepsPerVote; ++step) {
                // (1) at most one pop: an entry whose subtree cannot hold a closer hit any more is dropped and
                //     the lane pops again in the next step (bvh.h:221: far child only while best is farther).  An
                //     empty stack ends the light traversal (on into the scene BVH; best_t is still +inf) or the ray.
                {
                    const bool need = link == kLinkPop;
                    const bool has = need && sp > 0;
                    int32_t l = kLinkDone;
                    float t = -INFINITY;  // empty stack: t < best_t holds, link becomes l
                    if (has) {
                        --sp;
                        if (kSmemStack > 0 && sp < kSmemStack) {
                            top -= kExtendThreads;
                            RT_LD(top, l, t);
                        } else {
                            const float2 e = overflow[sp - kSmemStack];
                            l = __float_as_int(e.x);
                            t = e.y;
                        }
                    }
#if !RT_LIGHT_KERNEL
                    if (need && !has && lmode) {
                        lmode = false;
#if RT_EXT_SPLIT_NODES
                        node_base = bvh.q4lo;
#else
                        node_base = bvh.qnodes4;
#endif
                        l = scene_root;
                    }
#endif
                    if (need) link = t < best_t ? l : kLinkPop;
                }
                // (2) at most one node step: four slab tests, nearest child next, the others onto the stack
                if (link >= 0) {
                    auto push = [&](int32_t l, float t) {
                        if (kSmemStack > 0 && sp < kSmemStack) {
                            RT_ST(top, l, t);
                            top += kExtendThreads;
                        } else {
                            overflow[sp - kSmemStack] = make_float2(__int_as_float(l), t);
                        }
                        ++sp;
                    };
#if RT_EXT_SPLIT_NODES
                    const char *np = node_base + static_cast<size_t>(static_cast<uint32_t>(link)) * 32u;
                    const f8 na = ld8h<RT_EXT_NODE_L1>(np), nb = ld8h<RT_EXT_NODE_L1>(np + hi_off);  // grid, 6 plane words | 4 links
#else
                    const char *np = reinterpret_cast<const char *>(node_base + link);
                    const f8 na = ld8h<RT_EXT_NODE_L1>(np), nb = ld8h<RT_EXT_NODE_L1>(np + 32);  // 64 B node: grid, 6 plane words, 4 links
#endif
                    const Node4Test nt = qnode4_test(f2u(na.a), f2u(na.b), f2u(na.c), f2u(na.d), f2u(na.e), f2u(na.f), f2u(na.g),
                                                     f2u(na.h), f2u(nb.a), idir, o, one, eps, best_t);
                    float d0 = nt.d[0], d1 = nt.d[1], d2 = nt.d[2], d3 = nt.d[3];
                    int32_t l0 = static_cast<int32_t>(f2u(nb.b)), l1 = static_cast<int32_t>(f2u(nb.c));
                    int32_t l2 = static_cast<int32_t>(f2u(nb.d)), l3 = static_cast<int32_t>(f2u(nb.e));
                    // nearest child first, the others onto the stack farthest first (5-comparator network; ties keep
                    // the child order, the 4-wide image of "ties go left", bvh.h:216-219)
                    cswap(d0, l0, d1, l1);
                    cswap(d2, l2, d3, l3);
                    cswap(d0, l0, d2, l2);
                    cswap(d1, l1, d3, l3);
                    cswap(d1, l1, d2, l2);
                    // after the sort the hit children are d0..d(n-1); d1..d(n-1) go onto the stack so that d1 is
                    // on top: three predicated stores below the new top instead of three push sequences
                    const int n_push = (d1 < INFINITY ? 1 : 0) + (d2 < INFINITY ? 1 : 0) + (d3 < INFINITY ? 1 : 0);
                    if (kSmemStack > 0 && sp + n_push <= kSmemStack) {
                        uint2 *nt_top = top + n_push * kExtendThreads;
                        if (d1 < INFINITY) RT_ST(nt_top - 1 * kExtendThreads, l1, d1);
                        if (d2 < INFINITY) RT_ST(nt_top - 2 * kExtendThreads, l2, d2);
                        if (d3 < INFINITY) RT_ST(nt_top - 3 * kExtendThreads, l3, d3);
                        top = nt_top;
                        sp += n_push;
                    } else {  // rare: the shared part of the stack is full
                        if (d3 < INFINITY) push(l3, d3);
                        if (d2 < INFINITY) push(l2, d2);
                        if (d1 < INFINITY) push(l1, d1);
                    }
                    link = d0 < INFINITY ? l0 : kLinkPop;
                }
                // (3) postpone the first leaf and keep descending (the next step pops); a lane that meets a second
                //     one waits with it
                if (leaf == 0 && link_is_leaf(link)) {
                    leaf = link;
#if !RT_LIGHT_KERNEL
                    leaf_l = lmode;
#endif
                    link = kLinkPop;
                }
            }
        }

        // ---- leaf phase: all postponed leaves, two triangles per iteration -------------------------------
        {
            uint32_t k = static_cast<uint32_t>(~leaf);
            bool more = leaf != 0;
            while (__any_sync(FULL, more)) {
                if (more) {
                    const bool lt = leaf_l;
                    const char *p = reinterpret_cast<const char *>((lt ? lbvh.tris : bvh.tris) + k);
                    // intersect_ray_triangle, bvh.h:36-65 (same expression as tri_test() in pt_core.cuh with
                    // the reciprocal instead of the division)
                    auto tri = [&](const f8 &ta, const f4 &t2, uint32_t kk) {
                        const f3 e1 = mk3(ta.e, ta.f, ta.g), e2 = mk3(t2.x, t2.y, t2.z);
                        const f3 n = cross(e1, e2);
                        const f3 y = o - mk3(ta.a, ta.b, ta.c);
                        const f3 r = cross(d, y);
                        const float inv = rcp_rn(-dot(d, n));
                        const float beta = -dot(e2, r) * inv, gamma = dot(e1, r) * inv, t = dot(y, n) * inv;
                        if (beta >= 0.0f && gamma >= 0.0f && beta + gamma <= 1.0f && t >= eps && t < best_t) {
#if !RT_LIGHT_KERNEL
                            if (lt) {  // every hit counts, occluded or not, both faces (raytracer.h:79-84,255-261)
                                lsum += light_pdf_term(d, t, ld4(light_extra + kk));
                            } else
#endif
                            {
                                best_t = t;
                                best_b = beta;
                                best_c = gamma;
                                best_tri = static_cast<int32_t>(kk);
                            }
                        }
                        return (f2u(ta.d) & RT_LAST_BIT) != 0u;
                    };
                    // the second triangle is loaded speculatively (the array ends with a null triangle): the scene's
                    // leaves mostly hold a quad, and the load latency is paid once per leaf
                    const f8 ta = ld8h<RT_EXT_TRI_L1>(p), tb = ld8h<RT_EXT_TRI_L1>(p + 64);
                    const f4 ta2 = ld4h<RT_EXT_TRI_L1>(p + 32), tb2 = ld4h<RT_EXT_TRI_L1>(p + 96);
                    bool last = tri(ta, ta2, k);
                    if (!last) last = tri(tb, tb2, k + 1);
                    more = !last;
                    k += 2;
                }
            }
            leaf = 0;  // a lane that waited with a second leaf postpones it in step (3) of the next inner phase
        }
    }
}

// ---- k_lightpdf_list ----------------------------------------------------------------------------------
// bvh_mix_dist::pdf (raytracer.h:363-375) of the pending rays: an all-hit traversal of the light BVH (nothing is culled,
// the visiting order does not matter), result in q.lpdf.  As a traversal mode of k_extend (rounds 1 / 2) it cost 10.4 %
// of that kernel (16.3 of 156 ms per 256 spp): the few node steps of a light query went through the sorted,
// stack-based, leaf-postponing machinery of the closest-hit search, and cost k_extend three registers.  Now
//   * k_shade, when it queues a pending ray, tests it against the box of all lights (six planes): a miss gets
//     lpdf = 0 there and then, the others (33-50 % on config 4: every light-sampled direction passes) are listed
//     with a warp-aggregated append;
//   * k_lightpdf_list traverses the light BVH for the listed rays only, one thread per ray, unordered, with a stack of
//     links.
// Measured on config 4 per 256 spp: k_extend 156.1 -> 137.7 ms, k_lightpdf_list 6.0 ms, k_shade +1.7 ms.  A variant that
// scanned the whole queue in the light kernel (box test + CTA-level compaction there) took 11.2 ms: the scan is bound
// by the latency of its own record loads.
struct LightBox {
    float lo[3], hi[3];  // box of all light triangles with a margin (rt_gpu.cu, upload)
};
constexpr int kLightThreads = 256;

__device__ __forceinline__ float light_traverse(const DBvh &lbvh, const DLight *__restrict__ light_extra, f3 o, f3 d, f3 idir,
                                                float eps, uint32_t one) {
    int32_t stack[RT_EXT_STACK_CAP];  // the upload bounds the need of an unordered traversal as well (stack_need4)
    int sp = 0;
    float lsum = 0.0f;
    int32_t link = lbvh.root4;
    for (;;) {
        if (link >= 0) {
            const char *np = reinterpret_cast<const char *>(lbvh.qnodes4 + link);
            const f8 na = ld8(np), nb = ld8(np + 32);
            const Node4Test nt = qnode4_test(f2u(na.a), f2u(na.b), f2u(na.c), f2u(na.d), f2u(na.e), f2u(na.f), f2u(na.g), f2u(na.h),
                                             f2u(nb.a), idir, o, one, eps, INFINITY);
            const int32_t l[4] = {static_cast<int32_t>(f2u(nb.b)), static_cast<int32_t>(f2u(nb.c)), static_cast<int32_t>(f2u(nb.d)),
                                  static_cast<int32_t>(f2u(nb.e))};
            link = kLinkPop;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (nt.d[c] < INFINITY) {
                    if (link == kLinkPop) link = l[c];
                    else stack[sp++] = l[c];
                }
            }
        } else if (link != kLinkPop) {  // leaf: intersect_ray_triangle (bvh.h:36-65) on every triangle, every hit counts
            uint32_t k = static_cast<uint32_t>(~link);
            for (;;) {
                const char *p = reinterpret_cast<const char *>(lbvh.tris + k);
                const f8 ta = ld8(p);
                const f4 t2 = ld4(p + 32);
                const f3 e1 = mk3(ta.e, ta.f, ta.g), e2 = mk3(t2.x, t2.y, t2.z);
                const f3 n = cross(e1, e2);
                const f3 y = o - mk3(ta.a, ta.b, ta.c);
                const f3 r = cross(d, y);
                const float inv = rcp_rn(-dot(d, n));
                const float beta = -dot(e2, r) * inv, gamma = dot(e1, r) * inv, t = dot(y, n) * inv;
                if (beta >= 0.0f && gamma >= 0.0f && beta + gamma <= 1.0f && t >= eps && t < INFINITY)
                    lsum += light_pdf_term(d, t, ld4(light_extra + k));
                if (f2u(ta.d) & RT_LAST_BIT) break;
                ++k;
            }
            link = kLinkPop;
        }
        if (link == kLinkPop) {
            if (sp == 0) break;
            link = stack[--sp];
        }
    }
    return lsum;
}

// RT_LIGHT_KERNEL == 2: only the rays k_shade listed (those that pass the box of all lights).  The list index and the
// ray record of the next iteration are requested before the current ray is traversed (two dependent gathers from DRAM
// per ray: without the pipeline the kernel ran at a third of its instruction rate).
__global__ void __launch_bounds__(kLightThreads) k_lightpdf_list(DBvh lbvh, const DLight *__restrict__ light_extra, float inv_n_lights, float eps,
                                                                Queues q, uint32_t bounce, uint32_t one) {
    const uint32_t n = q.light_count[bounce * kCounterStride];
    const uint32_t stride = gridDim.x * kLightThreads;
    uint32_t j = blockIdx.x * kLightThreads + threadIdx.x;
    if (j >= n) return;
    uint32_t i_cur = __ldcs(q.light_list + j);
    uint32_t i_nxt = j + stride < n ? __ldcs(q.light_list + j + stride) : 0u;
    float4 d4 = q.d_in[i_cur], o4 = q.o_in[i_cur];
    for (;;) {
        const bool more = j + stride < n;
        float4 d4n = d4, o4n = o4;
        uint32_t i_nn = 0u;
        if (more) {
            d4n = q.d_in[i_nxt];
            o4n = q.o_in[i_nxt];
            if (j + 2u * stride < n) i_nn = __ldcs(q.light_list + j + 2u * stride);
        }
        const f3 o = mk3(o4.x, o4.y, o4.z), d = mk3(d4.x, d4.y, d4.z);
        const f3 idir = mk3(rcp_rn(d.x), rcp_rn(d.y), rcp_rn(d.z));
        q_store<0>(q.lpdf + i_cur, light_traverse(lbvh, light_extra, o, d, idir, eps, one) * inv_n_lights);
        if (!more) break;
        j += stride;
        i_cur = i_nxt;
        i_nxt = i_nn;
        d4 = d4n;
        o4 = o4n;
    }
}

// slab test of a ray against the box of all lights; NaNs (0 * inf) drop out of fminf / fmaxf: conservative
__device__ __forceinline__ bool light_box_test(const LightBox &box, f3 o, f3 d, float eps) {
    const float ix = rcp_rn(d.x), iy = rcp_rn(d.y), iz = rcp_rn(d.z);
    const float ax = (box.lo[0] - o.x) * ix, bx = (box.hi[0] - o.x) * ix;
    const float ay = (box.lo[1] - o.y) * iy, by = (box.hi[1] - o.y) * iy;
    const float az = (box.lo[2] - o.z) * iz, bz = (box.hi[2] - o.z) * iz;
    const float t0 = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), eps));
    const float t1 = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    return t0 <= t1;
}

// k_shade's warp-aggregated append to queue `next` (RT_LIGHT_KERNEL == 2): the lanes of `mask` (the warp's __ballot of
// the entries it keeps) get consecutive slots of the out queue, returned per lane.  A pending ray (`pend`) that misses
// the box of all lights has light pdf 0, stored at its slot of lpdf_out; the others are listed for k_lightpdf_list.
// Both atomics are issued before either result is waited for.  k_lightpdf_debug appends through here as well.
__device__ __forceinline__ uint32_t append_to_queue(const Queues &q, uint32_t *out_counter, uint32_t next, const LightBox &light_box,
                                                    uint32_t mask, bool pend, f3 o, f3 d, float eps) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = lane_id();
    uint32_t dst = 0;
    const bool pass = pend && light_box_test(light_box, o, d, eps);
    const uint32_t mp = __ballot_sync(FULL, pass);
    uint32_t lp = 0;
    if (lane == 0) {
        if (mask) dst = atomicAdd(out_counter, static_cast<uint32_t>(__popc(mask)));
        if (mp) lp = atomicAdd(q.light_count + next * kCounterStride, static_cast<uint32_t>(__popc(mp)));
    }
    dst = __shfl_sync(FULL, dst, 0) + static_cast<uint32_t>(__popc(mask & ((1u << lane) - 1u)));
    lp = __shfl_sync(FULL, lp, 0) + static_cast<uint32_t>(__popc(mp & ((1u << lane) - 1u)));
    if (pend && !pass) q_store<0>(q.lpdf_out + dst, 0.0f);
    if (pass) q.light_list[lp] = dst;
    return dst;
}

// rt_gpu_debug_light_pdf: n caller rays (o4 / d4, the pending bit set) appended as pending rays to queue 1 exactly as
// k_shade appends them; slot_of[i] = the queue slot of ray i.  Whole warps: the grid covers n rounded up to 32.
__global__ void __launch_bounds__(128) k_lightpdf_debug(const float4 *__restrict__ o4, const float4 *__restrict__ d4, uint32_t n, Queues q,
                                                       LightBox light_box, float eps, uint32_t *__restrict__ slot_of) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool alive = i < n;
    const float4 a = alive ? o4[i] : make_float4(0, 0, 0, 0), b = alive ? d4[i] : make_float4(0, 0, 1, 0);
    const f3 o = mk3(a.x, a.y, a.z), d = mk3(b.x, b.y, b.z);
    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, alive);
    const uint32_t dst = append_to_queue(q, q.count + kCounterStride, 1, light_box, mask, alive, o, d, eps);
    if (alive) {
        q.o_out[dst] = a;
        q.d_out[dst] = b;
        slot_of[i] = dst;
    }
}

// k_shade, bounce b.  For every entry of queue b:
//   1. if the path is pending (its previous bounce sampled a direction and the scene has lights): resolve that
//      bounce with the light pdf k_extend summed along this very ray — p = p_partial + (1 - VNDF_factor)/2 * lpdf,
//      p < EPS ends the path, else throughput = (thr * f_cos) / p  (shade_resolve, raytracer.h:572-590);
//   2. shade_begin: miss -> background; hit data; alpha coin; emission; strategy coin; direction sample;
//   3. shade_weights of the sampled direction (BRDF * cos, VNDF and cosine pdfs); without lights the bounce is
//      resolved at once, with lights the entry goes out pending;
//   4. survivors are compacted into queue b+1 with a warp-aggregated append.
// The light-pdf traversal itself lives in k_extend (second traversal mode of a pending ray).
#ifndef RT_SHADE_MINB
#define RT_SHADE_MINB 0
#endif
#ifndef RT_SHADE_PREFETCH
#define RT_SHADE_PREFETCH 1  // 0: off (38.25 ms per 256 spp); 1 (37.15): next iteration's queue records; 2: + its hit triangles / attributes; 3: + the radiance slot of a miss
#endif
__device__ __forceinline__ void pf_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#if RT_SHADE_MINB
__global__ void __launch_bounds__(kShadeThreads, RT_SHADE_MINB) k_shade(
#else
__global__ void __launch_bounds__(kShadeThreads) k_shade(
#endif
    DScene s, const float *__restrict__ lut_g, BatchParams bp, Queues q, uint32_t bounce_part, LightBox light_box) {
    __shared__ float lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = lut_g[i];
    __syncthreads();
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t part = bounce_part & ~(kPartFirst - 1u), bounce = bounce_part & (kPartFirst - 1u);
    const uint32_t count = part_end(part, q.count[bounce * kCounterStride]);  // this launch's part of the queue: [part_begin, count)
    uint32_t *const fetch_cursor = q.fetch_shade + bounce * kCounterStride;
    uint32_t *const out_counter = q.count + (bounce + 1) * kCounterStride;
    const bool last = bounce + 1 == s.ray_depth;
    const uint32_t lane = lane_id();
    uint32_t n_light = 0, n_shade = 0, n_ext = 0;
#if RT_SHADE_PREFETCH
    // Software pipeline of the work fetch: the cursor value of iteration k + 1 is requested during iteration k (its
    // atomic is in flight while the warp shades) and turned, half an iteration ahead of their use, into L1 prefetches
    // of the 32 queue records the warp will read next (and, level 2, into a look at their hit triangles, whose
    // DTri / DAttr lines are prefetched at the end of the iteration).
    uint32_t base_w = 0, ahead = 0;
    if (lane == 0) base_w = atomicAdd(fetch_cursor, 32u);
    base_w = __shfl_sync(FULL, base_w, 0) + part_begin(part, count);
    if (lane == 0) ahead = atomicAdd(fetch_cursor, 32u);
#endif
    for (;;) {
#if RT_SHADE_PREFETCH
        const uint32_t base = base_w;
#else
        uint32_t base = 0;  // the warp pulls the next 32 queue entries
        if (lane == 0) base = atomicAdd(fetch_cursor, 32u);
        base = __shfl_sync(FULL, base, 0) + part_begin(part, count);
#endif
        if (base >= count) break;
        const uint32_t i = base + lane;
        bool alive = false;
        f3 o = mk3(0, 0, 0), d = mk3(0, 0, 0), thr = mk3(0, 0, 0), rad = mk3(0, 0, 0);
        float pending = -1.0f;
        uint32_t pixel = 0, sample = 0;
        if (i < count) {
            const float4 o4 = q_load<1>(q.o_in + i), d4 = q_load<1>(q.d_in + i), t4 = q_load<1>(q.thr_in + i), h4 = q_load<1>(q.hit + i);
            o = mk3(o4.x, o4.y, o4.z);
            d = mk3(d4.x, d4.y, d4.z);
            thr = mk3(t4.x, t4.y, t4.z);
            pixel = __float_as_uint(o4.w);
            sample = __float_as_uint(d4.w) & 0x7FFFFFFFu;
            bool live = true;
#if RT_SHADE_PREFETCH >= 3
            if (__float_as_int(h4.w) < 0) pf_l1(q.rad + ((__float_as_uint(d4.w) & 0x7FFFFFFFu) - bp.s0) * bp.npix + (__float_as_uint(o4.w) - bp.pix0));  // a miss adds the background
#endif
            if (__float_as_uint(d4.w) >> 31) live = shade_resolve(s, thr, t4.w, q_load<1>(q.lpdf + i), thr);  // previous bounce
            if (live) {
                ++n_ext;  // this extension ray's hit is consumed (cast_ray of the reference)
                Hit h;
                h.t = h4.x;
                h.b = h4.y;
                h.c = h4.z;
                h.tri = __float_as_int(h4.w);
                const RngKey key{pixel, sample, bp.k0, bp.k1};
                n_shade += h.tri >= 0 ? 1u : 0u;
                ShadeMid mid;
                const f3 d_in = d;
                const ShadeStep step = shade_begin(s, lut, key, bounce, last, h, o, d, thr, rad, mid);
                alive = step == SHADE_PASS;
                if (step == SHADE_SAMPLED) {
                    n_light += s.n_lights > 0 ? 1u : 0u;  // bvh_mix_dist::pdf calls of the reference (raytracer.h:573)
                    const ShadeWeights w = shade_weights(s, mid, d_in);
                    if (len2(w.f_cos) != 0.0f) {  // raytracer.h:584-586
                        if (s.n_lights > 0) {  // resolved by the next k_shade with the light pdf of (pos, dir)
                            thr = thr * w.f_cos;
                            pending = w.p_partial;
                            alive = true;
                        } else {
                            alive = shade_resolve(s, thr * w.f_cos, w.p_partial, 0.0f, thr);
                        }
                        o = mid.pos;
                        d = mid.dir;
                    }
                }
                if (rad.x != 0.0f || rad.y != 0.0f || rad.z != 0.0f) {  // NaN != 0 is true: poisons the sample like the reference
                    const uint32_t slot = (sample - bp.s0) * bp.npix + (pixel - bp.pix0);
                    float4 acc = q_load<3>(q.rad + slot);
                    acc.x += rad.x;
                    acc.y += rad.y;
                    acc.z += rad.z;
                    q_store<3>(q.rad + slot, acc);
                }
            }
        }
#if RT_SHADE_PREFETCH
        // the next iteration's records -> L1; request the cursor value of the iteration after it
        base_w = __shfl_sync(FULL, ahead, 0) + part_begin(part, count);
        if (lane == 0) ahead = atomicAdd(fetch_cursor, 32u);
        const uint32_t i_next = base_w + lane;
#if RT_SHADE_PREFETCH >= 2
        int32_t tri_next = -1;
#endif
        if (i_next < count) {
            pf_l1(q.o_in + i_next);
            pf_l1(q.d_in + i_next);
            pf_l1(q.thr_in + i_next);
#if RT_SHADE_PREFETCH >= 2
            tri_next = __float_as_int(q.hit[i_next].w);
#else
            pf_l1(q.hit + i_next);
#endif
            if ((lane & 7u) == 0u) pf_l1(q.lpdf + i_next);
        }
#endif
        // warp-aggregated append: one atomicAdd per warp, slots handed out by __popc of the lower lanes
        const uint32_t mask = __ballot_sync(FULL, alive);
        uint32_t dst = 0;
#if RT_LIGHT_KERNEL == 2
        dst = append_to_queue(q, out_counter, bounce + 1, light_box, mask, alive && pending >= 0.0f, o, d, s.eps);
#else
        if (lane == 0 && mask) dst = atomicAdd(out_counter, static_cast<uint32_t>(__popc(mask)));
        dst = __shfl_sync(FULL, dst, 0) + static_cast<uint32_t>(__popc(mask & ((1u << lane) - 1u)));
#endif
        if (alive) {
            q_store<2>(q.o_out + dst, make_float4(o.x, o.y, o.z, __uint_as_float(pixel)));
            q_store<2>(q.d_out + dst, make_float4(d.x, d.y, d.z, __uint_as_float(sample | (pending >= 0.0f ? 0x80000000u : 0u))));
            q_store<2>(q.thr_out + dst, make_float4(thr.x, thr.y, thr.z, pending));
        }
#if RT_SHADE_PREFETCH >= 2
        if (tri_next >= 0) {
            pf_l1(s.scene.tris + tri_next);
            pf_l1(s.attrs + tri_next);
        }
#endif
    }
    // block-level reduction of the work counters -> one atomic per CTA and counter
    __shared__ uint32_t s_cnt[3];
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int off = 16; off > 0; off >>= 1) {
        n_light += __shfl_down_sync(0xFFFFFFFFu, n_light, off);
        n_shade += __shfl_down_sync(0xFFFFFFFFu, n_shade, off);
        n_ext += __shfl_down_sync(0xFFFFFFFFu, n_ext, off);
    }
    if (lane_id() == 0) {
        atomicAdd(&s_cnt[0], n_ext);
        atomicAdd(&s_cnt[1], n_light);
        atomicAdd(&s_cnt[2], n_shade);
    }
    __syncthreads();
    if (threadIdx.x < 3 && s_cnt[threadIdx.x]) atomicAdd(q.stats + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
}

// QNode4 records -> the two 32-byte-stride arrays k_extend reads (DBvh::q4lo); one thread per 16-byte quarter
__global__ void __launch_bounds__(256) k_split_nodes(const QNode4 *__restrict__ nodes, uint32_t n, char *__restrict__ lo, char *__restrict__ hi) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 4u) return;
    const uint32_t node = t >> 2, quarter = t & 3u;
    const uint4 v = reinterpret_cast<const uint4 *>(nodes)[t];
    char *dst = (quarter < 2 ? lo : hi) + static_cast<size_t>(node) * 32u + (quarter & 1u) * 16u;
    *reinterpret_cast<uint4 *>(dst) = v;
}

// sum_j sanitize(rad[j * npix + p]) over the k samples of a batch, j ascending.  MOMENTS also returns in .w the sum of
// y^2, y = (r + g + b) / 3 of each sanitised sample (the second moment of the adaptive stopping rule, adaptive.cuh).
template <bool MOMENTS>
__device__ __forceinline__ float4 sum_samples(const BatchParams &bp, const float4 *__restrict__ rad, uint32_t p) {
    f3 sum = mk3(0, 0, 0);
    float y2 = 0.0f;
    for (uint32_t j = 0; j < bp.k; ++j) {
        const float4 v = q_load<3>(rad + static_cast<size_t>(j) * bp.npix + p);
        const f3 c = sanitize(mk3(v.x, v.y, v.z));
        sum = sum + c;
        if (MOMENTS) {
            const float y = (c.x + c.y + c.z) / 3.0f;
            y2 += y * y;
        }
    }
    return make_float4(sum.x, sum.y, sum.z, y2);
}

// accum[pixel] += sum_j sanitize(rad[j * npix + p])  — fixed order, deterministic, no atomics
__global__ void __launch_bounds__(256) k_accumulate(BatchParams bp, const float4 *__restrict__ rad, float4 *__restrict__ accum) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= bp.npix) return;
    const float4 sum = sum_samples<false>(bp, rad, p);
    float4 a = accum[bp.pix0 + p];
    a.x += sum.x;
    a.y += sum.y;
    a.z += sum.z;
    accum[bp.pix0 + p] = a;
}

// RT_MODE_PRIMARY_IDS: hits of the pixel-centre rays (traced by k_extend like any other ray) -> scene.objects id
__global__ void __launch_bounds__(256) k_ids_from_hits(BatchParams bp, const float4 *__restrict__ hit, const DTri *__restrict__ tris,
                                                       int32_t *__restrict__ ids) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= bp.npix) return;
    const int32_t tri = __float_as_int(hit[p].w);
    ids[bp.pix0 + p] = tri < 0 ? -1 : static_cast<int32_t>(tris[tri].id_last & ~RT_LAST_BIT);
}

// rt_gpu_readback: packed rgb means = `res / samples` (raytracer.h:626), IEEE division like the host's
__global__ void __launch_bounds__(256) k_means(const float4 *__restrict__ accum, float samples, uint32_t n_pixels, float *__restrict__ rgb) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const float4 a = accum[p];
    rgb[static_cast<size_t>(p) * 3 + 0] = __fdiv_rn(a.x, samples);
    rgb[static_cast<size_t>(p) * 3 + 1] = __fdiv_rn(a.y, samples);
    rgb[static_cast<size_t>(p) * 3 + 2] = __fdiv_rn(a.z, samples);
}

// Device-side Image::set_pixel (image.h:40-82): mean -> ACES -> gamma 1/2.2 -> x255 -> clamp -> round
__device__ __forceinline__ void tonemap_pixel(float4 a, float samples, uint8_t *__restrict__ out) {
    const float c[3] = {a.x / samples, a.y / samples, a.z / samples};  // `res / samples`, raytracer.h:626
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float x = c[k];
        const float m = (x * (2.51f * x + 0.03f)) / (x * (2.43f * x + 0.59f) + 0.14f);
        const float v = powf(m, 1.0f / 2.2f) * 255.0f;
        const float cl = fminf(fmaxf(v, 0.0f), 255.0f);  // NaN -> 0
        out[k] = static_cast<uint8_t>(roundf(cl));
    }
}

__global__ void __launch_bounds__(256) k_tonemap(const float4 *__restrict__ accum, float samples, uint32_t n_pixels,
                                                 uint8_t *__restrict__ rgb8) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    tonemap_pixel(accum[p], samples, rgb8 + static_cast<size_t>(p) * 3);
}

// FP32 roofline probe: 16 independent FFMA chains per thread, no memory traffic.
__global__ void __launch_bounds__(256) k_fma_peak(float *out, float a, float b, int iters) {
    float x[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = static_cast<float>(threadIdx.x + i) * 1e-3f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = fmaf(x[i], a, b);
    }
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += x[i];
    if (s == 123.456f) out[0] = s;  // never true; keeps the chains alive
}

}  // namespace rt

#endif  // RT_KERNELS_CUH
