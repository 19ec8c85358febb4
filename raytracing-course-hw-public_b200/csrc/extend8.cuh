// extend8.cuh — k_extend over the 8-wide quantised nodes (QNode8, rt_types.h).
//
// Same job and same warp-synchronous phase structure as k_extend (kernels.cuh): closest hit per ray, for a
// "pending" ray first the all-hit traversal of the light BVH (bvh_mix_dist::pdf, raytracer.h:363-375); inner phase of
// predicated node steps behind a warp vote, leaf phase for the postponed triangles, per-lane ray refill from a
// warp-local block of queue entries.  What differs is the node step (Ylitie, Karras & Laine 2017, on this library's
// grid encoding):
//   * one step tests EIGHT child boxes (three 32-byte sectors) and yields an 8-bit hit mask;
//   * the children sit in octant-ordered slots, so the visiting order is `slot ^ octant of the ray`, highest first:
//     one 3-stage bit permutation of the mask per step instead of a distance sort of the children;
//   * the stack holds GROUPS (first inner child, permuted hit mask | imask) — at most one push per step — and no
//     distances: a stale entry is culled when its own children are tested against the current best_t.  On the bench
//     scene that is 10.1 node steps per path-traced ray against 16.0 of the 4-wide sorted traversal
//     (tools/wide_study.cpp), but ~300 instead of 216 instructions per step: measured 88 ms of k_extend8 against
//     83.7 ms of k_extend per 128 spp on the B200, which is why this build is optional (DESIGN.md, section 4);
//   * leaf children are (first triangle, hit slots | triangle counts) groups; one group per lane can be postponed, a
//     lane that meets a second one parks it as its current group and waits for the leaf phase.
// Group encoding (x, y):  y >= 2^24: node group, bits 24..31 = hit children by PRIORITY (bit p = slot p ^ octinv), bits
// 0..7 = the node's imask, x = index of its first inner child;  0 < y < 2^24: triangle group, bits 0..7 = hit leaf
// slots, bits 8..23 = the node's count field, x = the node's first triangle;  y == 0: nothing (x == kDone8: ray done).
#ifndef RT_EXTEND8_CUH
#define RT_EXTEND8_CUH

#include "kernels.cuh"

namespace rt {

#ifndef RT_EXT8_MINB
#define RT_EXT8_MINB 8
#endif
#ifndef RT_EXT8_MIN_SEARCH
#define RT_EXT8_MIN_SEARCH 16  // 16 / 20 / 24 -> 95.5 / 98.1 / 101.2 ms of k_extend8 per 128 spp
#endif
#ifndef RT_EXT8_STEPS_PER_VOTE
#define RT_EXT8_STEPS_PER_VOTE 2
#endif
#ifndef RT_EXT8_SMEM_STACK
#define RT_EXT8_SMEM_STACK 12
#endif
constexpr uint32_t kDone8 = 0xFFFFFFFFu;
constexpr uint32_t kRootGroup = 0x80000000u;  // "child 0 of base 0, imask 0" = node 0

__global__ void __launch_bounds__(kExtendThreads, RT_EXT8_MINB)
    k_extend8(DBvh bvh, DBvh lbvh, const DLight *__restrict__ light_extra, float inv_n_lights, float eps, Queues q, uint32_t bounce,
              uint32_t one) {
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t count = q.count[bounce * kCounterStride];
    const float4 *__restrict__ qo = q.o_in;
    const float4 *__restrict__ qd = q.d_in;
    uint32_t *cursor = q.fetch_ext + bounce * kCounterStride;
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;

    constexpr int kS = RT_EXT8_SMEM_STACK;
    __shared__ uint2 s_stack[kS * kExtendThreads];  // [entry][thread]: one 64-bit access per group
    uint2 overflow[2 * RT_STACK_SIZE - kS];  // at most two pushes per level of a tree no deeper than the binary one
    uint2 *top = s_stack + threadIdx.x;  // slot of the next push (valid while sp < kS)
    int sp = 0;
    uint32_t gx = kDone8, gy = 0;  // current group
    uint32_t tx = 0, ty = 0;       // postponed triangle group
    uint32_t ray = kNoRay;         // bit 31: pending (its light pdf is wanted)
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 1), idir = mk3(0, 0, 1);
    uint32_t octinv = 0;
    float best_t = INFINITY, best_b = 0.0f, best_c = 0.0f;
    int32_t best_tri = -1;
    bool lmode = false, leaf_l = false;
    float lsum = 0.0f;
    const QNode8 *node_base = bvh.qnodes8;
    const bool have_scene = bvh.n_nodes8 != 0, have_lights = lbvh.n_nodes8 != 0;
    uint32_t pool_next = 0, pool_end = 0;
    bool exhausted = false;

    auto push = [&](uint32_t x, uint32_t y) {
        if (sp < kS) {
            top[0] = make_uint2(x, y);
            top += kExtendThreads;
        } else {
            overflow[sp - kS] = make_uint2(x, y);
        }
        ++sp;
    };

    for (;;) {
        // ---- retire finished rays, refill idle lanes ---------------------------------------------------
        const bool idle = gy == 0 && gx == kDone8 && ty == 0;
        if (idle && ray != kNoRay) {
            const uint32_t r = ray & 0x7FFFFFFFu;
            if (ray >> 31) q_store<0>(q.lpdf + r, lsum * inv_n_lights);
            q_store<0>(q.hit + r, make_float4(best_t, best_b, best_c, __int_as_float(best_tri)));
            ray = kNoRay;
        }
        const uint32_t m_idle = __ballot_sync(FULL, idle);
        if (m_idle) {
            if (pool_next == pool_end && !exhausted) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(cursor, kRayBlock);
                base = __shfl_sync(FULL, base, 0);
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
                octinv = (idir.x < 0.0f ? 0u : 1u) | (idir.y < 0.0f ? 0u : 2u) | (idir.z < 0.0f ? 0u : 4u);
                best_t = INFINITY;
                best_b = best_c = 0.0f;
                best_tri = -1;
                sp = 0;
                top = s_stack + threadIdx.x;
                lsum = 0.0f;
                lmode = (__float_as_uint(d4.w) >> 31) != 0u && have_lights;
                ray |= __float_as_uint(d4.w) & 0x80000000u;
                node_base = lmode ? lbvh.qnodes8 : bvh.qnodes8;
                const bool any_root = lmode || have_scene;
                gx = any_root ? 0u : kDone8;
                gy = any_root ? kRootGroup : 0u;
            }
            pool_next += take;
            if (avail == 0 && m_idle == FULL) break;  // queue drained and nothing in flight
        }
        const bool can_refill = !exhausted || pool_next != pool_end;

        // ---- inner phase -------------------------------------------------------------------------------
        for (;;) {
            const bool done = gy == 0 && gx == kDone8;
            const uint32_t m_search = __ballot_sync(FULL, ty == 0 && !done);
            if (__popc(m_search) < RT_EXT8_MIN_SEARCH) {
                if (m_search == 0) break;
                if (__any_sync(FULL, ty != 0 || (can_refill && done))) break;
            }
#pragma unroll
            for (int step = 0; step < RT_EXT8_STEPS_PER_VOTE; ++step) {
                // (1) nothing in hand: next group from the stack; an empty stack ends the light traversal (on into the
                //     scene BVH, best_t is still +inf) or the ray
                if (gy == 0 && gx != kDone8) {
                    if (sp > 0) {
                        --sp;
                        if (sp < kS) {
                            top -= kExtendThreads;
                            const uint2 e = top[0];
                            gx = e.x;
                            gy = e.y;
                        } else {
                            const uint2 e = overflow[sp - kS];
                            gx = e.x;
                            gy = e.y;
                        }
                    } else if (lmode && have_scene) {
                        lmode = false;
                        node_base = bvh.qnodes8;
                        gx = 0u;
                        gy = kRootGroup;
                    } else {
                        lmode = false;
                        gx = kDone8;
                    }
                }
                // (2) a triangle group in hand: postpone it if this lane has none postponed yet, else wait
                if (gy != 0u && gy < 0x01000000u && ty == 0u) {
                    tx = gx;
                    ty = gy;
                    leaf_l = lmode;
                    gx = 0u;
                    gy = 0u;
                }
                // (3) a node group in hand: visit its first child in the ray's octant order
                if (gy >= 0x01000000u) {
                    const uint32_t p = bfind32(gy);
                    const uint32_t slot = (p - 24u) ^ octinv;
                    gy &= ~(1u << p);
                    const uint32_t child = gx + static_cast<uint32_t>(__popc(gy & 0xFFu & ((1u << slot) - 1u)));
                    if (gy >> 24) push(gx, gy);
                    const char *np = reinterpret_cast<const char *>(node_base + child);
                    const f8 h = ld8(np), ga = ld8(np + 32), gb = ld8(np + 64);
                    const Grid3 g = qgrid(f2u(h.a), f2u(h.b), f2u(h.c), idir, o);
                    const bool px = !(idir.x < 0.0f), py = !(idir.y < 0.0f), pz = !(idir.z < 0.0f);
                    const uint32_t hs =
                        q8_group_hits(f2u(ga.a), f2u(ga.b), f2u(ga.c), f2u(ga.d), f2u(ga.e), f2u(ga.f), g, px, py, pz, one, eps, best_t) |
                        q8_group_hits(f2u(gb.a), f2u(gb.b), f2u(gb.c), f2u(gb.d), f2u(gb.e), f2u(gb.f), g, px, py, pz, one, eps, best_t) << 4;
                    const uint32_t imask = f2u(h.d);
                    const uint32_t inner = hs & imask, leafm = hs & ~imask & leaf8_slots(f2u(h.g));  // no empty slot (leaf8_slots)
                    gx = inner ? f2u(h.e) : 0u;
                    gy = inner ? (oct_permute(inner, octinv) << 24) | imask : 0u;
                    if (leafm) {
                        const uint32_t ny = leafm | (f2u(h.g) << 8);
                        if (ty == 0u) {
                            tx = f2u(h.f);
                            ty = ny;
                            leaf_l = lmode;
                        } else {  // a second triangle group: park it in hand (the node group goes onto the stack) and wait
                            if (gy) push(gx, gy);
                            gx = f2u(h.f);
                            gy = ny;
                        }
                    }
                }
            }
        }

        // ---- leaf phase: the postponed triangle groups, leaf child by leaf child, two triangles per iteration ---
        {
            uint32_t k = 0;
            bool more = false;
            while (__any_sync(FULL, more || ty != 0u)) {
                if (!more && ty != 0u) {  // next hit leaf child of the group
                    const uint32_t s = bfind32(ty & 0xFFu);
                    k = tx + leaf8_offset(ty >> 8, s);
                    ty &= ~(1u << s);
                    if (!(ty & 0xFFu)) ty = 0u;
                    more = true;
                }
                if (more) {
                    const bool lt = leaf_l;
                    const char *p = reinterpret_cast<const char *>((lt ? lbvh.tris : bvh.tris) + k);
                    // intersect_ray_triangle, bvh.h:36-65 (tri_test() of pt_core.cuh with the reciprocal instead of the division)
                    auto tri = [&](const f8 &ta, const f4 &t2, uint32_t kk) {
                        const f3 e1 = mk3(ta.e, ta.f, ta.g), e2 = mk3(t2.x, t2.y, t2.z);
                        const f3 n = cross(e1, e2);
                        const f3 y = o - mk3(ta.a, ta.b, ta.c);
                        const f3 r = cross(d, y);
                        const float inv = rcp_rn(-dot(d, n));
                        const float beta = -dot(e2, r) * inv, gamma = dot(e1, r) * inv, t = dot(y, n) * inv;
                        if (beta >= 0.0f && gamma >= 0.0f && beta + gamma <= 1.0f && t >= eps && t < best_t) {
                            if (lt) {  // every hit counts, occluded or not, both faces (raytracer.h:79-84,255-261)
                                const f4 le = ld4(light_extra + kk);
                                const f3 xy = d * t;  // y - x
                                const float d2 = len2(xy);
                                const f3 w = xy * rsqrtf(d2);
                                lsum += d2 / (fabsf(dot(w, mk3(le.x, le.y, le.z))) * le.w);
                            } else {
                                best_t = t;
                                best_b = beta;
                                best_c = gamma;
                                best_tri = static_cast<int32_t>(kk);
                            }
                        }
                        return (f2u(ta.d) & RT_LAST_BIT) != 0u;
                    };
                    const f8 ta = ld8(p), tb = ld8(p + 64);  // the second one speculatively: the array ends with a null triangle
                    const f4 ta2 = ld4(p + 32), tb2 = ld4(p + 96);
                    bool last = tri(ta, ta2, k);
                    if (!last) last = tri(tb, tb2, k + 1);
                    more = !last;
                    k += 2;
                }
            }
        }
    }
}

}  // namespace rt

#endif  // RT_EXTEND8_CUH
