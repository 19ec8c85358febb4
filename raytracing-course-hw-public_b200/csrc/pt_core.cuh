// pt_core.cuh — per-ray / per-bounce device math of the wavefront path tracer.
//
// Everything here is a pure function of its arguments and is marked RT_HD so that the same source
// can also be compiled by the host compiler for unit tests of the math (tests/hostcheck); the
// kernels in kernels.cuh / extend8.cuh only add the queue plumbing.  Each function cites the reference code whose
// semantics it has to keep (Appendix B of SURVEY.md lists why each detail matters).
#ifndef RT_PT_CORE_CUH
#define RT_PT_CORE_CUH

#include <math.h>
#include <stdint.h>

#include "rt_types.h"

#if defined(__CUDACC__)
#define RT_HD __host__ __device__ __forceinline__
#define RT_D __device__ __forceinline__
#else
#define RT_HD inline
#define RT_D inline
#endif

namespace rt {

// ------------------------------------------------------------------------------------------------
// small vector types
// ------------------------------------------------------------------------------------------------
struct f3 {
    float x, y, z;
};
struct alignas(16) f4 {
    float x, y, z, w;
};

RT_HD f3 mk3(float x, float y, float z) { return f3{x, y, z}; }
RT_HD f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
RT_HD f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
RT_HD f3 operator*(f3 a, f3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
RT_HD f3 operator*(f3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_HD f3 operator*(float s, f3 a) { return mk3(a.x * s, a.y * s, a.z * s); }
RT_HD f3 operator-(f3 a) { return mk3(-a.x, -a.y, -a.z); }
RT_HD float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
RT_HD f3 cross(f3 a, f3 b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
RT_HD float len2(f3 a) { return dot(a, a); }
RT_HD f3 normalize(f3 a) { return a * (1.0f / sqrtf(len2(a))); }  // geometry::norm, geometry.h:31-34
// normalize_dir: for vectors that do NOT feed the GGX D term (geometric normal, sampled directions before the final
// half-vector): MUFU.RSQ instead of IEEE sqrt + division (a third of the instructions; `normalize` was 14 % of k_shade's).
// Everything the D term sees (shading normal, half vector, VNDF frame) keeps the IEEE form: with alpha = 0.0016
// near-mirrors D = alpha^2 / (pi (1 - ndh^2 + alpha^2 ndh^2)^2) amplifies a 1e-7 length error of ns or h to 10 % of D, and
// rsqrt everywhere biased the texall golden by 0.7 % at 131 072 spp (profiles/r2_normalize.md).
#if defined(__CUDA_ARCH__) && (!defined(RT_FAST_NORMALIZE) || RT_FAST_NORMALIZE)
RT_HD f3 normalize_dir(f3 a) { return a * rsqrtf(len2(a)); }
#else
RT_HD f3 normalize_dir(f3 a) { return normalize(a); }
#endif
// The same trade for the well-conditioned scalar divisions and square roots of the samplers, pdfs and the BRDF (MUFU.RCP /
// MUFU.SQRT, 1-2 ulp, instead of the IEEE sequences of ~9 instructions each): a relative error of 2e-7 in a factor of the
// estimator.  The host compilation (tests/hostcheck) keeps the IEEE forms.
#if defined(__CUDA_ARCH__) && (!defined(RT_FAST_SHADE_MATH) || RT_FAST_SHADE_MATH)
RT_HD float sh_div(float a, float b) { return __fdividef(a, b); }
RT_HD float sh_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
RT_HD float sh_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#else
RT_HD float sh_div(float a, float b) { return a / b; }
RT_HD float sh_rcp(float x) { return 1.0f / x; }
RT_HD float sh_sqrt(float x) { return sqrtf(x); }
#endif
RT_HD bool any_nan(f3 a) { return (a.x != a.x) || (a.y != a.y) || (a.z != a.z); }

#define RT_PI 3.14159265358979323846f
#define RT_INV_PI 0.31830988618379067154f

// 128-bit read-only loads (L1/L2 resident scene data)
#if defined(__CUDA_ARCH__)
RT_HD f4 ld4(const void *p) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(p));
    return f4{v.x, v.y, v.z, v.w};
}
RT_HD uint32_t ldu(const uint32_t *p) { return __ldg(p); }
#else
RT_HD f4 ld4(const void *p) { return *reinterpret_cast<const f4 *>(p); }
RT_HD uint32_t ldu(const uint32_t *p) { return *p; }
#endif

// 256-bit read-only load (LDG.E.256 on sm_100a; needs a 32-byte aligned address): one L1 tag lookup per
// lane instead of two.  The traversal is bound by L1TEX wavefronts (one per distinct 128 B line per load
// instruction), so halving the number of load instructions per node is what matters.
struct alignas(32) f8 {
    float a, b, c, d, e, f, g, h;
};
#if defined(__CUDA_ARCH__)
RT_HD f8 ld8(const void *p) {
    f8 v;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(v.a), "=f"(v.b), "=f"(v.c), "=f"(v.d), "=f"(v.e), "=f"(v.f), "=f"(v.g), "=f"(v.h)
        : "l"(p));
    return v;
}
#else
RT_HD f8 ld8(const void *p) { return *reinterpret_cast<const f8 *>(p); }
#endif

RT_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
#endif
}
RT_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 keyed (pixel, sample, 2*bounce + block); replaces std::minstd_rand seeded per span
// (raytracer.h:456-489, 646-648).  Lane assignment per bounce (<= 6 uniforms, SURVEY Appendix B.11):
//   block 0: [0] alpha coin  [1] strategy coin  [2] vndf u1 | mixture selector  [3] vndf u2 | light index
//   block 1: [0],[1] cosine (z, phi) | light point (u, v)
//   counter word 2 = 0xFFFFFFFF: [0],[1] pixel jitter
// ------------------------------------------------------------------------------------------------
RT_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return static_cast<uint32_t>((static_cast<uint64_t>(a) * b) >> 32);
#endif
}

struct u4 {
    uint32_t x, y, z, w;
};

RT_HD u4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return u4{c0, c1, c2, c3};
}
RT_HD float u01(uint32_t bits) { return static_cast<float>(bits >> 8) * (1.0f / 16777216.0f); }  // [0,1)

struct RngKey {
    uint32_t pixel, sample, k0, k1;
};
RT_HD u4 rng_block(const RngKey &k, uint32_t bounce, uint32_t block) {
    return philox4x32_10(k.pixel, k.sample, 2u * bounce + block, 0u, k.k0, k.k1);
}
RT_HD u4 rng_jitter(const RngKey &k) { return philox4x32_10(k.pixel, k.sample, 0xFFFFFFFFu, 0u, k.k0, k.k1); }

// ------------------------------------------------------------------------------------------------
// camera: gen_ray, raytracer.h:516-538; fov_y from Camera::fov_y, scene.h:69-71 (host-computed tans)
// ------------------------------------------------------------------------------------------------
struct Camera {
    f3 pos, right, up, fwd;
    float tan_half_x, tan_half_y;
    float inv_w2, inv_h2;  // 2/width, 2/height
};

RT_HD f3 camera_dir(const Camera &c, float px, float py) {
    const float a = (px * c.inv_w2 - 1.0f) * c.tan_half_x;
    const float b = (py * c.inv_h2 - 1.0f) * c.tan_half_y;
    return normalize(a * c.right - b * c.up + c.fwd);
}

// ------------------------------------------------------------------------------------------------
// intersection primitives (src/bvh.h)
// ------------------------------------------------------------------------------------------------
struct Hit {
    float t, b, c;  // distance and the barycentrics of vertex b and c (xs.z, xs.x, xs.y of bvh.h:45-47)
    int32_t tri;    // BVH-order triangle index, -1 = miss
};

// intersect(ray, aabb, min_dst), bvh.h:137-152 with the division replaced by a multiplication with
// 1/dir.  Returns the entry distance max(t_min, min_dst) or a negative value on a miss.
RT_HD float slab(float lox, float loy, float loz, float hix, float hiy, float hiz, f3 o, f3 idir, float min_dst) {
    const float x0 = (lox - o.x) * idir.x, x1 = (hix - o.x) * idir.x;
    const float y0 = (loy - o.y) * idir.y, y1 = (hiy - o.y) * idir.y;
    const float z0 = (loz - o.z) * idir.z, z1 = (hiz - o.z) * idir.z;
    const float tmin = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fminf(z0, z1));
    const float tmax = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fmaxf(z0, z1));
    return (tmin <= tmax && tmax >= min_dst) ? fmaxf(tmin, min_dst) : -1.0f;
}

// intersect_ray_triangle + intersect(ray, triangle, min_dst), bvh.h:36-65 (Cramer's rule written as
// scalar triple products).  Accept iff beta >= 0, gamma >= 0, beta + gamma <= 1, t >= min_dst.
RT_HD bool tri_test(f3 a, f3 e1, f3 e2, f3 o, f3 d, float min_dst, float &t, float &beta, float &gamma) {
    const f3 n = cross(e1, e2);
    const float det = -dot(d, n);
    const f3 y = o - a;
    const f3 r = cross(d, y);
    const float inv = 1.0f / det;
    beta = -dot(e2, r) * inv;
    gamma = dot(e1, r) * inv;
    t = dot(y, n) * inv;
    return beta >= 0.0f && gamma >= 0.0f && beta + gamma <= 1.0f && t >= min_dst;
}

// ---- quantised 2-wide node (QNode, rt_types.h): both child slab tests from one 32-byte record.  Host checks only
// (the device traversed this form before the 4-wide one); qplane() below is shared by all node widths. --------------
// Plane byte q of a word -> the float 1 + q * 2^-16 (q added into mantissa bits 7..14), so that
//   t(q) = (org + q * cell - o) / d = fma(1 + q * 2^-16, A, B)   with  A = 2^16 * cell / d,  B = (org - o) / d - A
// costs one byte-dot-product + one FFMA per plane and no integer->float conversion.  The extraction is a DP4A
// (`one + byte_K(w) * 0x80`), not a byte permute: k_extend is bound by the ALU pipe (PRMT / FMNMX / SEL: 67 % of
// peak against 25 % for the FMA pipe, profiles/r1_v10_k_extend_ncu_full.csv), and IDP.4A issues on the FMA pipe.
// A is 256 x the node's extent in ray space, so B carries an absolute rounding error of ~2^-8 cell; the packer
// keeps a 1/64-cell margin for it.
// `one` = 0x3F800000, which k_extend receives as a kernel ARGUMENT so that it stays in a register.
template <int K> RT_HD float qplane(uint32_t w, uint32_t one) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(__dp4a(w, 0x80u << (8 * K), one));
#else
    return u2f(one + (((w >> (8 * K)) & 255u) << 7));
#endif
}
RT_HD uint32_t qnode_one() { return 0x3F800000u; }  // the kernel gets it as an argument instead

struct NodeTest {
    float dl, dr;  // entry distances (clipped to eps from below)
    bool hl, hr;
};

// Per-ray byte selectors: identity where the ray runs in the positive direction of the axis, min<->max swapped
// where it runs in the negative one; applied to a plane word they give (left.near, left.far, right.near, right.far).
struct RaySwz {
    uint32_t x, y, z;
};
RT_HD RaySwz ray_swizzle(f3 idir) {
    RaySwz r;
    r.x = idir.x < 0.0f ? 0x2301u : 0x3210u;
    r.y = idir.y < 0.0f ? 0x2301u : 0x3210u;
    r.z = idir.z < 0.0f ? 0x2301u : 0x3210u;
    return r;
}
RT_HD uint32_t swz(uint32_t w, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, sel);
#else
    return sel == 0x3210u ? w : (((w & 0x00FF00FFu) << 8) | ((w >> 8) & 0x00FF00FFu));
#endif
}

RT_HD NodeTest qnode_test(const uint32_t ox, const uint32_t oy, const uint32_t oz, const uint32_t q0, const uint32_t q1,
                          const uint32_t q2, f3 idir, f3 o, RaySwz sw, uint32_t one, float eps, float best_t) {
    // ray-space planes as in qnode4_test: subtract the ray origin before the multiply
    const float ax = u2f((ox << 23) + 0x08000000u) * idir.x, bx = fmaf(u2f(ox) - o.x, idir.x, -ax);
    const float ay = u2f((oy << 23) + 0x08000000u) * idir.y, by = fmaf(u2f(oy) - o.y, idir.y, -ay);
    const float az = u2f((oz << 23) + 0x08000000u) * idir.z, bz = fmaf(u2f(oz) - o.z, idir.z, -az);
    const uint32_t wx = swz(q0, sw.x), wy = swz(q1, sw.y), wz = swz(q2, sw.z);
    // slab test of both children (bvh.h:137-152): entry = max of the three near planes, exit = min of the three far
    // planes, interval clipped to [eps, best_t] (hit <=> entry <= exit): visits the boxes
    // `t_min <= t_max && t_max >= eps && max(t_min, eps) < best` does, plus harmless ties with best_t.  A ray parallel
    // to a slab gives NaN or +-inf planes; fmaxf/fminf drop the NaNs: conservative.
    NodeTest r;
    r.dl = fmaxf(fmaxf(fmaxf(fmaf(qplane<0>(wx, one), ax, bx), fmaf(qplane<0>(wy, one), ay, by)), fmaf(qplane<0>(wz, one), az, bz)), eps);
    const float el = fminf(fminf(fminf(fmaf(qplane<1>(wx, one), ax, bx), fmaf(qplane<1>(wy, one), ay, by)), fmaf(qplane<1>(wz, one), az, bz)), best_t);
    r.dr = fmaxf(fmaxf(fmaxf(fmaf(qplane<2>(wx, one), ax, bx), fmaf(qplane<2>(wy, one), ay, by)), fmaf(qplane<2>(wz, one), az, bz)), eps);
    const float er = fminf(fminf(fminf(fmaf(qplane<3>(wx, one), ax, bx), fmaf(qplane<3>(wy, one), ay, by)), fmaf(qplane<3>(wz, one), az, bz)), best_t);
    r.hl = r.dl <= el;
    r.hr = r.dr <= er;
    return r;
}

// closest_hit() over the quantised nodes, in the kernel's arithmetic (1/d once, fused o/d) — the sequential
// statement of what k_extend computes per ray; the host tests compare its hits with closest_hit()'s.
RT_HD Hit closest_hit_q(const DBvh &bvh, f3 o, f3 d, float min_dst, uint32_t *steps = nullptr) {
    Hit best;
    best.t = INFINITY;
    best.b = best.c = 0.0f;
    best.tri = -1;
    if (bvh.root == RT_LINK_NONE) return best;
    const f3 idir = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    const RaySwz sw = ray_swizzle(idir);
    int32_t stack_link[RT_STACK_SIZE];
    float stack_t[RT_STACK_SIZE];
    int sp = 0;
    int32_t link = bvh.root;
    for (;;) {
        if (link >= 0) {
            if (steps) ++*steps;
            const f8 nq = ld8(bvh.qnodes + link);
            const NodeTest nt = qnode_test(f2u(nq.a), f2u(nq.b), f2u(nq.c), f2u(nq.d), f2u(nq.e), f2u(nq.f), idir, o, sw,
                                           qnode_one(), min_dst, best.t);
            const int32_t ll = static_cast<int32_t>(f2u(nq.g)), lr = static_cast<int32_t>(f2u(nq.h));
            if (nt.hl || nt.hr) {
                const bool right_first = nt.hr && (!nt.hl || nt.dl > nt.dr);
                link = right_first ? lr : ll;
                if (nt.hl && nt.hr) {
                    stack_link[sp] = right_first ? ll : lr;
                    stack_t[sp] = right_first ? nt.dl : nt.dr;
                    ++sp;
                }
                continue;
            }
        } else {
            uint32_t k = static_cast<uint32_t>(~link);
            for (;;) {
                const char *p = reinterpret_cast<const char *>(bvh.tris + k);
                const f4 t0 = ld4(p), t1 = ld4(p + 16), t2 = ld4(p + 32);
                float t, b, c;
                if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), o, d, min_dst, t, b,
                             c) &&
                    t < best.t) {
                    best.t = t;
                    best.b = b;
                    best.c = c;
                    best.tri = static_cast<int32_t>(k);
                }
                if (f2u(t0.w) & RT_LAST_BIT) break;
                ++k;
            }
        }
        for (;;) {
            if (sp == 0) return best;
            --sp;
            if (stack_t[sp] < best.t) {
                link = stack_link[sp];
                break;
            }
        }
    }
}

// ---- 4-wide quantised node (QNode4): four slab tests from one 64-byte record ------------------------------------
// near/far plane words are picked per axis by the sign of the ray direction (a register select, no byte permute);
// d[c] = entry distance of child c clipped to eps from below, or +inf when the child is missed.
struct Node4Test {
    float d[4];
};
// RT_EXT_FFMA2 (device only): the 24 plane evaluations of a node step as 12 packed FFMA2 (fma.rn.f32x2, sm_100+: two
// IEEE fused multiply-adds per instruction with the scale and offset as broadcast scalar operands) — the same 24
// results bit for bit, half the FMA issue slots of the slab tests.
#ifndef RT_EXT_FFMA2
#define RT_EXT_FFMA2 1
#endif
// the four plane distances of one plane word: t[c] = fma(1 + byte_c(w) * 2^-16, a, b)
RT_HD void q4_axis(uint32_t w, float a, float b, uint32_t one, float t[4]) {
#if defined(__CUDA_ARCH__) && RT_EXT_FFMA2
    unsigned long long q01, q23, r01, r23, aa, bb;
    asm("mov.b64 %0, {%1, %2};" : "=l"(q01) : "f"(qplane<0>(w, one)), "f"(qplane<1>(w, one)));
    asm("mov.b64 %0, {%1, %2};" : "=l"(q23) : "f"(qplane<2>(w, one)), "f"(qplane<3>(w, one)));
    asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
    asm("mov.b64 %0, {%1, %1};" : "=l"(bb) : "f"(b));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r01) : "l"(q01), "l"(aa), "l"(bb));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r23) : "l"(q23), "l"(aa), "l"(bb));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(t[0]), "=f"(t[1]) : "l"(r01));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(t[2]), "=f"(t[3]) : "l"(r23));
#else
    t[0] = fmaf(qplane<0>(w, one), a, b);
    t[1] = fmaf(qplane<1>(w, one), a, b);
    t[2] = fmaf(qplane<2>(w, one), a, b);
    t[3] = fmaf(qplane<3>(w, one), a, b);
#endif
}
RT_HD Node4Test qnode4_test(const uint32_t ox, const uint32_t oy, const uint32_t oz, const uint32_t lox, const uint32_t loy,
                            const uint32_t loz, const uint32_t hix, const uint32_t hiy, const uint32_t hiz, f3 idir, f3 o,
                            uint32_t one, float eps, float best_t) {
    // plane t = (org + q * cell - o) / d = fma(1 + q * 2^-16, ax, bx).  The grid origin is subtracted from the ray origin
    // BEFORE the multiply (bvh.h:137-152 does the same), so the rounding error of bx is relative to |org - o|, the
    // ray's distance to the node.  The former fma(org, 1/d, -o * (1/d)) rounded o * (1/d) first: an error relative to
    // |o| itself, which outgrew the packer's 1/64-cell margin for small nodes ~1e3 of their extent away from the world
    // origin, and those nodes lost hits.  Same instruction count (FADD + FFMA instead of FFMA + FADD per axis).
    const float ax = u2f((ox << 23) + 0x08000000u) * idir.x, bx = fmaf(u2f(ox) - o.x, idir.x, -ax);
    const float ay = u2f((oy << 23) + 0x08000000u) * idir.y, by = fmaf(u2f(oy) - o.y, idir.y, -ay);
    const float az = u2f((oz << 23) + 0x08000000u) * idir.z, bz = fmaf(u2f(oz) - o.z, idir.z, -az);
    const bool px = !(idir.x < 0.0f), py = !(idir.y < 0.0f), pz = !(idir.z < 0.0f);
    const uint32_t nx = px ? lox : hix, fx = px ? hix : lox;
    const uint32_t ny = py ? loy : hiy, fy = py ? hiy : loy;
    const uint32_t nz = pz ? loz : hiz, fz = pz ? hiz : loz;
    float tnx[4], tny[4], tnz[4], tfx[4], tfy[4], tfz[4];
    q4_axis(nx, ax, bx, one, tnx);
    q4_axis(ny, ay, by, one, tny);
    q4_axis(nz, az, bz, one, tnz);
    q4_axis(fx, ax, bx, one, tfx);
    q4_axis(fy, ay, by, one, tfy);
    q4_axis(fz, az, bz, one, tfz);
    Node4Test r;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 4; ++c) {
        const float entry = fmaxf(fmaxf(fmaxf(tnx[c], tny[c]), tnz[c]), eps);
        const float exit_ = fminf(fminf(fminf(tfx[c], tfy[c]), tfz[c]), best_t);
        r.d[c] = entry <= exit_ ? entry : INFINITY;
    }
    return r;
}
// compare-exchange of (distance, link) pairs, ascending by distance; equal distances keep their order (ties: lower
// child index first, the 4-wide image of "ties go left", bvh.h:216-219)
RT_HD void cswap(float &da, int32_t &la, float &db, int32_t &lb) {
    const bool sw = db < da;
    const float td = sw ? db : da, ud = sw ? da : db;
    const int32_t tl = sw ? lb : la, ul = sw ? la : lb;
    da = td; db = ud; la = tl; lb = ul;
}

// closest_hit() over the 4-wide nodes (sequential statement of k_extend's 4-wide mode); `steps` counts node steps.
RT_HD Hit closest_hit_q4(const DBvh &bvh, f3 o, f3 d, float min_dst, uint32_t *steps) {
    Hit best;
    best.t = INFINITY;
    best.b = best.c = 0.0f;
    best.tri = -1;
    if (bvh.root4 == RT_LINK_NONE) return best;
    const f3 idir = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    int32_t stack_link[RT_STACK_SIZE * 2];
    float stack_t[RT_STACK_SIZE * 2];
    int sp = 0;
    int32_t link = bvh.root4;
    for (;;) {
        if (link >= 0) {
            if (steps) ++*steps;
            const char *p = reinterpret_cast<const char *>(bvh.qnodes4 + link);
            const f8 na = ld8(p), nb = ld8(p + 32);
            const Node4Test nt = qnode4_test(f2u(na.a), f2u(na.b), f2u(na.c), f2u(na.d), f2u(na.e), f2u(na.f), f2u(na.g),
                                             f2u(na.h), f2u(nb.a), idir, o, qnode_one(), min_dst, best.t);
            float d0 = nt.d[0], d1 = nt.d[1], d2 = nt.d[2], d3 = nt.d[3];
            int32_t l0 = static_cast<int32_t>(f2u(nb.b)), l1 = static_cast<int32_t>(f2u(nb.c));
            int32_t l2 = static_cast<int32_t>(f2u(nb.d)), l3 = static_cast<int32_t>(f2u(nb.e));
            cswap(d0, l0, d1, l1);
            cswap(d2, l2, d3, l3);
            cswap(d0, l0, d2, l2);
            cswap(d1, l1, d3, l3);
            cswap(d1, l1, d2, l2);
            if (d3 < INFINITY) { stack_link[sp] = l3; stack_t[sp++] = d3; }
            if (d2 < INFINITY) { stack_link[sp] = l2; stack_t[sp++] = d2; }
            if (d1 < INFINITY) { stack_link[sp] = l1; stack_t[sp++] = d1; }
            if (d0 < INFINITY) {
                link = l0;
                continue;
            }
        } else {
            uint32_t k = static_cast<uint32_t>(~link);
            for (;;) {
                const char *p = reinterpret_cast<const char *>(bvh.tris + k);
                const f4 t0 = ld4(p), t1 = ld4(p + 16), t2 = ld4(p + 32);
                float t, b, c;
                if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), o, d, min_dst, t, b,
                             c) &&
                    t < best.t) {
                    best.t = t;
                    best.b = b;
                    best.c = c;
                    best.tri = static_cast<int32_t>(k);
                }
                if (f2u(t0.w) & RT_LAST_BIT) break;
                ++k;
            }
        }
        for (;;) {
            if (sp == 0) return best;
            --sp;
            if (stack_t[sp] < best.t) {
                link = stack_link[sp];
                break;
            }
        }
    }
}

// ---- 8-wide quantised node (QNode8, rt_types.h): eight slab tests from one 96-byte record ----------------------------
RT_HD uint32_t bfind32(uint32_t x) {  // index of the highest set bit (x != 0)
#if defined(__CUDA_ARCH__)
    return 31u - static_cast<uint32_t>(__clz(static_cast<int>(x)));
#else
    return 31u - static_cast<uint32_t>(__builtin_clz(x));
#endif
}
RT_HD uint32_t popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return static_cast<uint32_t>(__popc(x));
#else
    return static_cast<uint32_t>(__builtin_popcount(x));
#endif
}
// octinv: bit k set where the ray runs in the POSITIVE direction of axis k.  A child in slot s (bit k set = positive
// side along axis k) is visited in the order of decreasing s ^ octinv: near side first along every axis.
RT_HD uint32_t ray_octinv(f3 d) { return (d.x < 0.0f ? 0u : 1u) | (d.y < 0.0f ? 0u : 2u) | (d.z < 0.0f ? 0u : 4u); }
// bit s of m -> bit s ^ octinv
RT_HD uint32_t oct_permute(uint32_t m, uint32_t octinv) {
    if (octinv & 1u) m = ((m & 0x55u) << 1) | ((m >> 1) & 0x55u);
    if (octinv & 2u) m = ((m & 0x33u) << 2) | ((m >> 2) & 0x33u);
    if (octinv & 4u) m = ((m & 0x0Fu) << 4) | ((m >> 4) & 0x0Fu);
    return m;
}
struct Grid3 {
    float ax, bx, ay, by, az, bz;
};
RT_HD Grid3 qgrid(uint32_t ox, uint32_t oy, uint32_t oz, f3 idir, f3 o) {  // ray-space grid as in qnode4_test
    Grid3 g;
    g.ax = u2f((ox << 23) + 0x08000000u) * idir.x, g.bx = fmaf(u2f(ox) - o.x, idir.x, -g.ax);
    g.ay = u2f((oy << 23) + 0x08000000u) * idir.y, g.by = fmaf(u2f(oy) - o.y, idir.y, -g.ay);
    g.az = u2f((oz << 23) + 0x08000000u) * idir.z, g.bz = fmaf(u2f(oz) - o.z, idir.z, -g.az);
    return g;
}
// slab test of child C of a plane group: entry (max of the near planes, eps) <= exit (min of the far planes, best_t)
template <int C> RT_HD bool q4_hit(uint32_t nx, uint32_t ny, uint32_t nz, uint32_t fx, uint32_t fy, uint32_t fz, const Grid3 &g, uint32_t one,
                                   float eps, float best_t) {
    const float entry = fmaxf(fmaxf(fmaxf(fmaf(qplane<C>(nx, one), g.ax, g.bx), fmaf(qplane<C>(ny, one), g.ay, g.by)),
                                    fmaf(qplane<C>(nz, one), g.az, g.bz)), eps);
    const float exit_ = fminf(fminf(fminf(fmaf(qplane<C>(fx, one), g.ax, g.bx), fmaf(qplane<C>(fy, one), g.ay, g.by)),
                                    fmaf(qplane<C>(fz, one), g.az, g.bz)), best_t);
    return entry <= exit_;
}
// hit bits of the four children of one plane group (lo x/y/z, hi x/y/z words)
RT_HD uint32_t q8_group_hits(uint32_t lox, uint32_t loy, uint32_t loz, uint32_t hix, uint32_t hiy, uint32_t hiz, const Grid3 &g, bool px,
                             bool py, bool pz, uint32_t one, float eps, float best_t) {
    const uint32_t nx = px ? lox : hix, fx = px ? hix : lox;
    const uint32_t ny = py ? loy : hiy, fy = py ? hiy : loy;
    const uint32_t nz = pz ? loz : hiz, fz = pz ? hiz : loz;
    return (q4_hit<0>(nx, ny, nz, fx, fy, fz, g, one, eps, best_t) ? 1u : 0u) | (q4_hit<1>(nx, ny, nz, fx, fy, fz, g, one, eps, best_t) ? 2u : 0u) |
           (q4_hit<2>(nx, ny, nz, fx, fy, fz, g, one, eps, best_t) ? 4u : 0u) | (q4_hit<3>(nx, ny, nz, fx, fy, fz, g, one, eps, best_t) ? 8u : 0u);
}
// triangle position of the leaf child in slot s: tri_base + the counts (2 bits per slot) of the lower slots
RT_HD uint32_t leaf8_offset(uint32_t counts, uint32_t s) {
    const uint32_t below = counts & ((1u << (2u * s)) - 1u);
    return popc32(below & 0x5555u) + 2u * popc32(below & 0xAAAAu);
}
// bit s set where slot s is a leaf child (count != 0).  An empty slot's inverted box is not always a miss: an axis-parallel
// ray has 1/d = +-inf on the other two axes, their slab planes become NaN and drop out of fminf / fmaxf, and in a node
// that is flat along the ray the remaining axis' planes 0 and 255 can coincide.  Its leaf8_offset is the next slot's
// first triangle, so a hit empty slot visits triangles twice: harmless for a closest hit, a doubled light-pdf term.
RT_HD uint32_t leaf8_slots(uint32_t counts) {
    uint32_t m = (counts | (counts >> 1)) & 0x5555u;
    m = (m | (m >> 1)) & 0x3333u;
    m = (m | (m >> 2)) & 0x0F0Fu;
    return (m | (m >> 4)) & 0xFFu;
}

// closest_hit() over the 8-wide nodes: the sequential statement of k_extend's 8-wide mode (group stack without
// distances: an entry is culled when its own children are tested against the current best).  `steps` counts node steps.
RT_HD Hit closest_hit_q8(const DBvh &bvh, f3 o, f3 d, float min_dst, uint32_t *steps) {
    Hit best;
    best.t = INFINITY;
    best.b = best.c = 0.0f;
    best.tri = -1;
    if (bvh.n_nodes8 == 0) return best;
    const f3 idir = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    const bool px = !(idir.x < 0.0f), py = !(idir.y < 0.0f), pz = !(idir.z < 0.0f);
    const uint32_t octinv = (px ? 1u : 0u) | (py ? 2u : 0u) | (pz ? 4u : 0u);
    uint32_t sx[RT_STACK_SIZE], sy[RT_STACK_SIZE];
    int sp = 0;
    uint32_t gx = 0, gy = 0x80000000u;  // pseudo group: "child 0 of nothing" = the root
    for (;;) {
        if (gy >> 24) {
            const uint32_t p = bfind32(gy);
            const uint32_t slot = (p - 24u) ^ octinv;
            gy &= ~(1u << p);
            const uint32_t child = gx + popc32(gy & 0xFFu & ((1u << slot) - 1u));
            if (gy >> 24) {
                sx[sp] = gx;
                sy[sp++] = gy;
            }
            if (steps) ++*steps;
            const char *np = reinterpret_cast<const char *>(bvh.qnodes8 + child);
            const f8 h = ld8(np), a = ld8(np + 32), b = ld8(np + 64);
            const Grid3 g = qgrid(f2u(h.a), f2u(h.b), f2u(h.c), idir, o);
            const uint32_t hs = q8_group_hits(f2u(a.a), f2u(a.b), f2u(a.c), f2u(a.d), f2u(a.e), f2u(a.f), g, px, py, pz, qnode_one(), min_dst, best.t) |
                                q8_group_hits(f2u(b.a), f2u(b.b), f2u(b.c), f2u(b.d), f2u(b.e), f2u(b.f), g, px, py, pz, qnode_one(), min_dst, best.t) << 4;
            const uint32_t imask = f2u(h.d), counts = f2u(h.g);
            uint32_t leaf = hs & ~imask & leaf8_slots(counts);
            while (leaf) {  // highest slot first, like the kernel's leaf phase
                const uint32_t s = bfind32(leaf);
                leaf &= ~(1u << s);
                uint32_t k = f2u(h.f) + leaf8_offset(counts, s);
                for (;;) {
                    const char *tp = reinterpret_cast<const char *>(bvh.tris + k);
                    const f4 t0 = ld4(tp), t1 = ld4(tp + 16), t2 = ld4(tp + 32);
                    float t, bb, cc;
                    if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), o, d, min_dst, t, bb, cc) && t < best.t) {
                        best.t = t;
                        best.b = bb;
                        best.c = cc;
                        best.tri = static_cast<int32_t>(k);
                    }
                    if (f2u(t0.w) & RT_LAST_BIT) break;
                    ++k;
                }
            }
            gx = f2u(h.e);
            gy = (oct_permute(hs & imask, octinv) << 24) | (imask & 0xFFu);
            if (gy >> 24) continue;
        }
        if (sp == 0) return best;
        --sp;
        gx = sx[sp];
        gy = sy[sp];
    }
}

struct TravCounters {
    uint32_t nodes, tris;
};

// BVH::intersect_ray, bvh.h:170-235, iteratively: near child first (ties: left first, bvh.h:216),
// far child visited only while the best hit is farther than its entry distance (bvh.h:221),
// strictly-closer-wins / first-found-wins-ties (bvh.h:132).
RT_HD Hit closest_hit(const DBvh &bvh, f3 o, f3 d, float min_dst) {
    Hit best;
    best.t = INFINITY;
    best.b = best.c = 0.0f;
    best.tri = -1;
    if (bvh.root == RT_LINK_NONE) return best;
    const f3 idir = mk3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    int32_t stack_link[RT_STACK_SIZE];
    float stack_t[RT_STACK_SIZE];
    int sp = 0;
    int32_t link = bvh.root;
    for (;;) {
        if (link >= 0) {
            const char *p = reinterpret_cast<const char *>(bvh.nodes + link);
            const f8 na = ld8(p), nb = ld8(p + 32);
            const f4 n0 = f4{na.a, na.b, na.c, na.d}, n1 = f4{na.e, na.f, na.g, na.h};
            const f4 n2 = f4{nb.a, nb.b, nb.c, nb.d}, n3 = f4{nb.e, nb.f, nb.g, nb.h};
            const float dl = slab(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, o, idir, min_dst);
            const float dr = slab(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, o, idir, min_dst);
            const int32_t ll = static_cast<int32_t>(f2u(n3.x)), lr = static_cast<int32_t>(f2u(n3.y));
            const bool hl = dl >= 0.0f && dl < best.t, hr = dr >= 0.0f && dr < best.t;
            if (hl && hr) {
                const bool swap = dl > dr;
                stack_link[sp] = swap ? ll : lr;
                stack_t[sp] = swap ? dl : dr;
                ++sp;
                link = swap ? lr : ll;
                continue;
            }
            if (hl || hr) {
                link = hl ? ll : lr;
                continue;
            }
        } else {
            uint32_t k = static_cast<uint32_t>(~link);
            for (;;) {
                const char *p = reinterpret_cast<const char *>(bvh.tris + k);
                const f4 t0 = ld4(p), t1 = ld4(p + 16), t2 = ld4(p + 32);
                float t, b, c;
                if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), o, d, min_dst, t, b,
                             c) &&
                    t < best.t) {
                    best.t = t;
                    best.b = b;
                    best.c = c;
                    best.tri = static_cast<int32_t>(k);
                }
                if (f2u(t0.w) & RT_LAST_BIT) break;
                ++k;
            }
        }
        // pop, skipping subtrees that can no longer contain a closer hit
        for (;;) {
            if (sp == 0) return best;
            --sp;
            if (stack_t[sp] < best.t) {
                link = stack_link[sp];
                break;
            }
        }
    }
}

// bvh_mix_dist::pdf, raytracer.h:363-375: ALL hits along (x, dir) with t >= eps, occluded or not,
// both faces; each contributes |y - x|^2 / (|dir . n_y| * area) (raytracer.h:79-84,255-261);
// the sum is divided by the number of lights.  BVH::foreach_intersection, bvh.h:237-260.
// the same sum over the 8-wide light BVH (every node whose box the ray meets, every triangle hit)
RT_HD float light_pdf_q8(const DScene &s, f3 x, f3 dir) {
    const DBvh &bvh = s.light;
    const f3 idir = mk3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);
    const bool px = !(idir.x < 0.0f), py = !(idir.y < 0.0f), pz = !(idir.z < 0.0f);
    uint32_t sx[RT_STACK_SIZE], sy[RT_STACK_SIZE];
    int sp = 0;
    uint32_t gx = 0, gy = 0x80000000u;
    float sum = 0.0f;
    for (;;) {
        if (gy >> 24) {
            const uint32_t p = bfind32(gy);
            const uint32_t slot = p - 24u;  // no ordering needed: all hits count
            gy &= ~(1u << p);
            const uint32_t child = gx + popc32(gy & 0xFFu & ((1u << slot) - 1u));
            if (gy >> 24) {
                sx[sp] = gx;
                sy[sp++] = gy;
            }
            const char *np = reinterpret_cast<const char *>(bvh.qnodes8 + child);
            const f8 h = ld8(np), a = ld8(np + 32), b = ld8(np + 64);
            const Grid3 g = qgrid(f2u(h.a), f2u(h.b), f2u(h.c), idir, x);
            const uint32_t hs = q8_group_hits(f2u(a.a), f2u(a.b), f2u(a.c), f2u(a.d), f2u(a.e), f2u(a.f), g, px, py, pz, qnode_one(), s.eps, INFINITY) |
                                q8_group_hits(f2u(b.a), f2u(b.b), f2u(b.c), f2u(b.d), f2u(b.e), f2u(b.f), g, px, py, pz, qnode_one(), s.eps, INFINITY) << 4;
            const uint32_t imask = f2u(h.d), counts = f2u(h.g);
            uint32_t leaf = hs & ~imask & leaf8_slots(counts);
            while (leaf) {
                const uint32_t sl = bfind32(leaf);
                leaf &= ~(1u << sl);
                uint32_t k = f2u(h.f) + leaf8_offset(counts, sl);
                for (;;) {
                    const char *tp = reinterpret_cast<const char *>(bvh.tris + k);
                    const f4 t0 = ld4(tp), t1 = ld4(tp + 16), t2 = ld4(tp + 32);
                    float t, bb, cc;
                    if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), x, dir, s.eps, t, bb, cc)) {
                        const f4 le = ld4(s.light_extra + k);
                        const f3 xy = dir * t;  // y - x, as light_pdf forms it
                        const float d2 = len2(xy);
                        const f3 w = xy * (1.0f / sqrtf(d2));
                        sum += d2 / (fabsf(dot(w, mk3(le.x, le.y, le.z))) * le.w);
                    }
                    if (f2u(t0.w) & RT_LAST_BIT) break;
                    ++k;
                }
            }
            gx = f2u(h.e);
            gy = ((hs & imask) << 24) | (imask & 0xFFu);
            if (gy >> 24) continue;
        }
        if (sp == 0) break;
        --sp;
        gx = sx[sp];
        gy = sy[sp];
    }
    return sum / static_cast<float>(s.n_lights);
}

RT_HD float light_pdf(const DScene &s, f3 x, f3 dir) {
    const DBvh &bvh = s.light;
    if (bvh.n_nodes8 != 0) return light_pdf_q8(s, x, dir);
    if (bvh.root == RT_LINK_NONE) return 0.0f;
    const f3 idir = mk3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);
    int32_t stack_link[RT_STACK_SIZE];
    int sp = 0;
    int32_t link = bvh.root;
    float sum = 0.0f;
    for (;;) {
        if (link >= 0) {
            const char *p = reinterpret_cast<const char *>(bvh.nodes + link);
            const f8 na = ld8(p), nb = ld8(p + 32);
            const f4 n0 = f4{na.a, na.b, na.c, na.d}, n1 = f4{na.e, na.f, na.g, na.h};
            const f4 n2 = f4{nb.a, nb.b, nb.c, nb.d}, n3 = f4{nb.e, nb.f, nb.g, nb.h};
            const bool hl = slab(n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, x, idir, s.eps) >= 0.0f;
            const bool hr = slab(n1.z, n1.w, n2.x, n2.y, n2.z, n2.w, x, idir, s.eps) >= 0.0f;
            const int32_t ll = static_cast<int32_t>(f2u(n3.x)), lr = static_cast<int32_t>(f2u(n3.y));
            if (hl && hr) {
                stack_link[sp++] = lr;
                link = ll;
                continue;
            }
            if (hl || hr) {
                link = hl ? ll : lr;
                continue;
            }
        } else {
            uint32_t k = static_cast<uint32_t>(~link);
            for (;;) {
                const char *p = reinterpret_cast<const char *>(bvh.tris + k);
                const f4 t0 = ld4(p), t1 = ld4(p + 16), t2 = ld4(p + 32);
                float t, b, c;
                if (tri_test(mk3(t0.x, t0.y, t0.z), mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z), x, dir, s.eps, t, b,
                             c)) {
                    const f4 le = ld4(s.light_extra + k);
                    // y - x = dir * t, as the kernels form it (light_pdf_term).  The reference's (x + dir * t) - x loses
                    // the low bits of t * dir to the magnitude of x: 4 % of a term at |x| = 3e4 and t = 0.1.
                    const f3 xy = dir * t;
                    const float d2 = len2(xy);
                    const f3 w = xy * (1.0f / sqrtf(d2));
                    sum += d2 / (fabsf(dot(w, mk3(le.x, le.y, le.z))) * le.w);
                }
                if (f2u(t0.w) & RT_LAST_BIT) break;
                ++k;
            }
        }
        if (sp == 0) break;
        link = stack_link[--sp];
    }
    return sum / static_cast<float>(s.n_lights);
}

// ------------------------------------------------------------------------------------------------
// textures + materials (src/geometry.h:517-631) and hit shading data (to_intersection_info, bvh.h:80-121)
// ------------------------------------------------------------------------------------------------
// Texture::sample: repeat wrap, texel = (int)(u*W) without half-texel offset, bilinear with wrapped
// neighbours, per-texel gamma BEFORE interpolation (LUT == powf(k/255, 2.2f)), alpha untouched;
// 1-texel textures are returned raw (geometry.h:548-550).
// One out-of-line copy on the device (k_shade calls it for up to four maps per hit): 5 % less k_shade time than the
// four inlined copies (code size / instruction cache), measured on the B200.
#if defined(__CUDACC__) && !defined(RT_TEX_INLINE)
__host__ __device__ __noinline__
#else
RT_HD
#endif
f4 tex_sample(const DScene &s, const float *lut, int32_t tex, float u, float v, bool gamma) {
    const f4 ti = ld4(s.textures + tex);
    const uint32_t off = f2u(ti.x), w = f2u(ti.y), h = f2u(ti.z);
    const float k255 = 1.0f / 255.0f;
    if (w * h == 1u) {
        const uint32_t p = ldu(s.texels + off);
        return f4{(p & 255u) * k255, ((p >> 8) & 255u) * k255, ((p >> 16) & 255u) * k255, (p >> 24) * k255};
    }
    const float tx = (u - floorf(u)) * static_cast<float>(w);
    const float ty = (v - floorf(v)) * static_cast<float>(h);
    uint32_t x0 = static_cast<uint32_t>(static_cast<int>(tx)), y0 = static_cast<uint32_t>(static_cast<int>(ty));
    x0 = x0 < w ? x0 : w - 1;  // u - floor(u) can round to 1.0f
    y0 = y0 < h ? y0 : h - 1;
    const float dx = tx - static_cast<float>(x0), dy = ty - static_cast<float>(y0);
    const uint32_t x1 = (x0 == w - 1) ? 0u : x0 + 1, y1 = (y0 == h - 1) ? 0u : y0 + 1;  // mod_inc, geometry.h:521
    const uint32_t p00 = ldu(s.texels + off + x0 + y0 * w), p01 = ldu(s.texels + off + x0 + y1 * w);
    const uint32_t p10 = ldu(s.texels + off + x1 + y0 * w), p11 = ldu(s.texels + off + x1 + y1 * w);
    const float wx0 = 1.0f - dx, wy0 = 1.0f - dy;
    f4 r;
    if (gamma) {
#define RT_BIL(sh) (wx0 * (wy0 * lut[(p00 >> sh) & 255u] + dy * lut[(p01 >> sh) & 255u]) + \
                    dx * (wy0 * lut[(p10 >> sh) & 255u] + dy * lut[(p11 >> sh) & 255u]))
        r.x = RT_BIL(0);
        r.y = RT_BIL(8);
        r.z = RT_BIL(16);
#undef RT_BIL
    } else {
#define RT_BIL(sh) (wx0 * (wy0 * (((p00 >> sh) & 255u) * k255) + dy * (((p01 >> sh) & 255u) * k255)) + \
                    dx * (wy0 * (((p10 >> sh) & 255u) * k255) + dy * (((p11 >> sh) & 255u) * k255)))
        r.x = RT_BIL(0);
        r.y = RT_BIL(8);
        r.z = RT_BIL(16);
#undef RT_BIL
    }
    r.w = wx0 * (wy0 * ((p00 >> 24) * k255) + dy * ((p01 >> 24) * k255)) +
          dx * (wy0 * ((p10 >> 24) * k255) + dy * ((p11 >> 24) * k255));
    return r;
}

// Scene::bg_at, scene.h:83-89: bg_color * bg.sample((x, y), 2.2) with the equirectangular coordinates
// x = 0.5 + 0.5 atan2(d.z, d.x) / pi, y = 0.5 - asin(d.y) / pi.  At HEAD `bg` is the 1x1 white texture (USE_ENV_MAP =
// false, config.h:36), i.e. the constant bg_color: env_tex < 0.
RT_HD f3 bg_at(const DScene &s, const float *lut, f3 d) {
    const f3 bg = mk3(s.bg[0], s.bg[1], s.bg[2]);
    if (s.env_tex < 0) return bg;
    const float x = 0.5f + 0.5f * atan2f(d.z, d.x) * RT_INV_PI;
    const float y = 0.5f - asinf(d.y) * RT_INV_PI;
    const f4 c = tex_sample(s, lut, s.env_tex, x, y, true);
    return bg * mk3(c.x, c.y, c.z);
}

// ray_intersection_info, bvh.h:18-29 (normals already flipped towards the ray, bvh.h:111-112)
struct Surface {
    f3 ng, ns;     // geometric / shading normal
    f3 color;      // base colour rgb
    float alpha;   // base colour alpha (coverage)
    f3 emission;
    float metallic, roughness, ior;
};

RT_HD Surface make_surface(const DScene &s, const float *lut, const Hit &h, f3 dir) {
    Surface sf;
    const char *tp = reinterpret_cast<const char *>(s.scene.tris + h.tri);
    const f4 t1 = ld4(tp + 16), t2 = ld4(tp + 32);
    const char *ap = reinterpret_cast<const char *>(s.attrs + h.tri);
    const f8 aa = ld8(ap), ab = ld8(ap + 32);
    const f4 a0 = f4{aa.a, aa.b, aa.c, aa.d}, a1 = f4{aa.e, aa.f, aa.g, aa.h};
    const f4 a2 = f4{ab.a, ab.b, ab.c, ab.d}, a3 = f4{ab.e, ab.f, ab.g, ab.h};
    f3 ng = normalize_dir(cross(mk3(t1.x, t1.y, t1.z), mk3(t2.x, t2.y, t2.z)));  // Object::base_normal
    const bool inside = dot(ng, dir) > 0.0f;                                   // bvh.h:92
    const float w0 = 1.0f - h.b - h.c;                                         // triangle::interop, geometry.h:497-502
    f3 smooth = normalize(mk3(a0.x, a0.y, a0.z) * w0 + mk3(a1.x, a1.y, a1.z) * h.b + mk3(a2.x, a2.y, a2.z) * h.c);
    if (dot(ng, smooth) < 0.0f) smooth = -smooth;  // bvh.h:95-97
    const float tu = a0.w * w0 + a2.w * h.b + a3.y * h.c;
    const float tv = a1.w * w0 + a3.x * h.b + a3.z * h.c;
    const char *mp = reinterpret_cast<const char *>(s.materials + f2u(a3.w));
    const f8 ma = ld8(mp), mb = ld8(mp + 32);
    const f4 m0 = f4{ma.a, ma.b, ma.c, ma.d}, m1 = f4{ma.e, ma.f, ma.g, ma.h};
    const f4 m2 = f4{mb.a, mb.b, mb.c, mb.d}, m3 = f4{mb.e, mb.f, mb.g, mb.h};
    const int32_t color_tex = static_cast<int32_t>(f2u(m2.z)), emissive_tex = static_cast<int32_t>(f2u(m2.w));
    const int32_t mr_tex = static_cast<int32_t>(f2u(m3.x)), normal_tex = static_cast<int32_t>(f2u(m3.y));

    f3 ns = smooth;
    if (normal_tex >= 0) {  // default NORMAL_UP decodes to (0,0,1): shading normal = smooth normal
        f3 tangent = mk3(1.0f, 0.0f, 0.0f);
        if (s.tangents) {
            const char *gp = reinterpret_cast<const char *>(s.tangents + h.tri);
            const f4 g0 = ld4(gp), g1 = ld4(gp + 16), g2 = ld4(gp + 32);
            tangent = normalize(mk3(g0.x, g0.y, g0.z) * w0 + mk3(g0.w, g1.x, g1.y) * h.b + mk3(g1.z, g1.w, g2.x) * h.c);
        }
        const f3 bitangent = cross(smooth, tangent);  // not normalised, bvh.h:102
        const f4 n01 = tex_sample(s, lut, normal_tex, tu, tv, false);
        const f3 nl = normalize(mk3(n01.x * 2.0f - 1.0f, n01.y * 2.0f - 1.0f, n01.z * 2.0f - 1.0f));
        ns = normalize(nl.x * tangent + nl.y * bitangent + nl.z * smooth);
    } else if (s.tangents) {
        // (0,0,1) in a frame whose z is `smooth`: still the smooth normal
        ns = smooth;
    }
    sf.ng = inside ? -ng : ng;
    sf.ns = inside ? -ns : ns;

    f4 col = f4{m0.x, m0.y, m0.z, m0.w};
    if (color_tex >= 0) {
        const f4 c = tex_sample(s, lut, color_tex, tu, tv, true);
        col = f4{col.x * c.x, col.y * c.y, col.z * c.z, col.w * c.w};
    }
    sf.color = mk3(col.x, col.y, col.z);
    sf.alpha = col.w;
    sf.emission = mk3(m1.x, m1.y, m1.z);
    if (emissive_tex >= 0) {
        const f4 e = tex_sample(s, lut, emissive_tex, tu, tv, true);
        sf.emission = sf.emission * mk3(e.x, e.y, e.z);
    }
    sf.roughness = m1.w;
    sf.metallic = m2.x;
    if (mr_tex >= 0) {
        const f4 mr = tex_sample(s, lut, mr_tex, tu, tv, false);
        sf.metallic *= mr.z;   // metallic = B, roughness = G (geometry.h:623-626)
        sf.roughness *= mr.y;
    }
    sf.ior = m2.y;
    return sf;
}

// ------------------------------------------------------------------------------------------------
// sampling distributions (src/raytracer.h:86-262) and BRDF (raytracer.h:264-343)
// ------------------------------------------------------------------------------------------------
RT_HD void sincos_2pi(float u, float &s, float &c) {  // sin/cos(2*pi*u)
#if defined(__CUDA_ARCH__)
    sincospif(2.0f * u, &s, &c);
#else
    s = sinf(2.0f * RT_PI * u);
    c = cosf(2.0f * RT_PI * u);
#endif
}

RT_HD f3 choose_local_x(f3 n) {  // VNDF_dist::choose_local_x, raytracer.h:208-219
    f3 r = mk3(1.0f, 1.0f, 1.0f);
    const float dn = n.x + n.y + n.z;
    // one well-conditioned division (|n.k| > 0.5, or the largest component): MUFU.RCP leaves the frame orthogonal to
    // 2e-7 instead of 6e-8; the normalisation stays IEEE (the frame feeds the D term of vndf_pdf)
    if (fabsf(n.x) > 0.5f) r.x -= sh_div(dn, n.x);
    else if (fabsf(n.y) > 0.5f) r.y -= sh_div(dn, n.y);
    else r.z -= sh_div(dn, n.z);
    return normalize(r);
}

// VNDF_dist::sample (Heitz 2018), raytracer.h:140-173. alpha = max(roughness, MIN_ROUGHNESS)^2.
RT_HD f3 vndf_sample(float alpha, f3 in_dir, f3 ns, f3 nx, float u1, float u2) {  // nx = choose_local_x(ns)
    const f3 ny = cross(ns, nx);
    const f3 v = -normalize_dir(mk3(dot(nx, in_dir), dot(ny, in_dir), dot(ns, in_dir)));
    const f3 vh = normalize_dir(mk3(alpha * v.x, alpha * v.y, v.z));
    const float lensq = vh.x * vh.x + vh.y * vh.y;
    const f3 T1 = lensq > 0.0f ? mk3(-vh.y, vh.x, 0.0f) * sh_rcp(sh_sqrt(lensq)) : mk3(1.0f, 0.0f, 0.0f);
    const f3 T2 = cross(vh, T1);
    const float r = sh_sqrt(u1);
    float sp, cp;
    sincos_2pi(u2, sp, cp);
    const float t1 = r * cp;
    float t2 = r * sp;
    const float sh = 0.5f * (1.0f + vh.z);
    t2 = (1.0f - sh) * sh_sqrt(1.0f - t1 * t1) + sh * t2;
    const float t3 = sh_sqrt(fmaxf(0.0f, 1.0f - t1 * t1 - t2 * t2));
    const f3 nh = t1 * T1 + t2 * T2 + t3 * vh;
    const f3 ne = normalize_dir(mk3(alpha * nh.x, alpha * nh.y, fmaxf(0.0f, nh.z)));
    const f3 res_n = normalize_dir(ne.x * nx + ne.y * ny + ne.z * ns);  // the half vector is re-normalised (IEEE) by the caller
    return in_dir - res_n * (2.0f * dot(in_dir, res_n));  // geometry::reflect
}

// VNDF_dist::pdf, raytracer.h:175-206
// nx = choose_local_x(ns), hw = normalize(dir - in_dir): both are shared with the sampler / the BRDF by the caller
RT_HD float vndf_pdf(float alpha, float eps, f3 in_dir, f3 ns, f3 nx, f3 hw) {
    const f3 ny = cross(ns, nx);
    const f3 v = -mk3(dot(nx, in_dir), dot(ny, in_dir), dot(ns, in_dir));
    const f3 n = mk3(dot(nx, hw), dot(ny, hw), dot(ns, hw));
    const float vdn = dot(v, n);
    if (!(vdn > 0.0f)) return 0.0f;
    const float ax = v.x * alpha, ay = v.y * alpha;
    const float lambda = (-1.0f + sh_sqrt(1.0f + sh_div(ax * ax + ay * ay, v.z * v.z))) * 0.5f;
    const float g1 = sh_rcp(1.0f + lambda);
    const float nxa = sh_div(n.x, alpha), nya = sh_div(n.y, alpha);
    const float q = nxa * nxa + nya * nya + n.z * n.z;
    const float dn = sh_div(RT_INV_PI, alpha * alpha * q * q);
    // g1 * vdn * dn / max(eps, v.z) / 4 / vdn
    return sh_div(sh_div(g1 * vdn * dn, fmaxf(eps, v.z)) * 0.25f, vdn);
}

// cosine_dist::sample = norm(n + uniform_sphere), sphere from z in U[-1,1], phi in U[0,2pi) (raytracer.h:94-121)
RT_HD f3 cosine_sample(f3 ng, float u1, float u2) {
    const float z = u1 * 2.0f - 1.0f;
    const float cz = sh_sqrt(fmaxf(0.0f, 1.0f - z * z));
    float sp, cp;
    sincos_2pi(u2, sp, cp);
    return normalize_dir(ng + mk3(cz * cp, cz * sp, z));
}
RT_HD float cosine_pdf(f3 ng, f3 dir) { return fmaxf(dot(ng, dir) * RT_INV_PI, 0.0f); }  // raytracer.h:123-128

// bvh_mix_dist::sample -> triangle_dist::sample, raytracer.h:227-239,355-361: uniform light index,
// (u,v) folded, p = A + (B-A)*v + (C-A)*u.
RT_HD f3 light_sample(const DScene &s, f3 x, float u_index, float u, float v) {
    uint32_t k = static_cast<uint32_t>(u_index * static_cast<float>(s.n_lights));
    k = k < s.n_lights ? k : s.n_lights - 1;
    const char *p = reinterpret_cast<const char *>(s.light_sample + k);
    const f4 t0 = ld4(p), t1 = ld4(p + 16), t2 = ld4(p + 32);
    if (u + v > 1.0f) {
        u = 1.0f - u;
        v = 1.0f - v;
    }
    const f3 pt = mk3(t0.x, t0.y, t0.z) + mk3(t1.x, t1.y, t1.z) * v + mk3(t2.x, t2.y, t2.z) * u;
    return normalize_dir(pt - x);
}

RT_HD float pow5(float x) {
    const float x2 = x * x;
    return x * x2 * x2;
}

// specular_brdf = V * D, raytracer.h:273-293
RT_HD float specular_brdf(float alpha, f3 in_dir, f3 out_dir, f3 ns, f3 h) {
    const float a2 = alpha * alpha;
    const float ndh = dot(ns, h);
    const float dd = ndh * ndh * (a2 - 1.0f) + 1.0f;
    const float d = sh_div((ndh > 0.0f ? a2 : 0.0f) * RT_INV_PI, dd * dd);  // the division is well-conditioned; dd is not (normalize)
    const float ndo = dot(ns, out_dir), ndi = -dot(ns, in_dir);
    const float div1 = fabsf(ndo) + sh_sqrt(a2 + (1.0f - a2) * ndo * ndo);
    const float div2 = fabsf(ndi) + sh_sqrt(a2 + (1.0f - a2) * ndi * ndi);
    const float vis = (dot(h, out_dir) > 0.0f && -dot(h, in_dir) > 0.0f) ? sh_rcp(div1 * div2) : 0.0f;
    return vis * d;
}

// pbr_brdf, raytracer.h:295-343: (1-m) * mix(diffuse c/pi, spec, F(ior)) + m * spec * (c + (1-c) F5)
RT_HD f3 pbr_brdf(const Surface &sf, float alpha, f3 in_dir, f3 out_dir, f3 h) {  // h = halfway, raytracer.h:131-134
    const float spec = specular_brdf(alpha, in_dir, out_dir, sf.ns, h);
    const float p5 = pow5(1.0f - fabsf(dot(-in_dir, h)));
    f3 res = mk3(0.0f, 0.0f, 0.0f);
    if (sf.metallic < 1.0f) {
        const float r0 = sh_div(1.0f - sf.ior, 1.0f + sf.ior);
        const float f0 = r0 * r0;
        const float fr = f0 + (1.0f - f0) * p5;
        const f3 diel = sf.color * (RT_INV_PI * (1.0f - fr)) + mk3(spec, spec, spec) * fr;
        res = res + (1.0f - sf.metallic) * diel;
    }
    if (sf.metallic > 0.0f) {
        const f3 f = mk3(sf.color.x + (1.0f - sf.color.x) * p5, sf.color.y + (1.0f - sf.color.y) * p5,
                         sf.color.z + (1.0f - sf.color.z) * p5);
        res = res + sf.metallic * (spec * f);
    }
    return res;
}

// ------------------------------------------------------------------------------------------------
// one bounce of shade(), raytracer.h:555-591, as a state transition of an iterative path:
//   radiance += throughput * (what this hit returns when the recursion below it is 0)
//   throughput *= scl  (raytracer.h:580-590)
// Returns true when the path continues with (o, d).
// ------------------------------------------------------------------------------------------------
// The bounce is split in two so that the kernel can run the light-pdf traversal of all 32 lanes as ONE
// warp-synchronous loop between the halves (k_shade); shade_bounce() below is the plain composition.
struct ShadeMid {
    Surface sf;
    f3 pos, dir;
    f3 nx;  // VNDF frame axis choose_local_x(ns): one evaluation serves the sampler and the pdf
    float alpha;
};
enum ShadeStep { SHADE_END = 0, SHADE_PASS = 1, SHADE_SAMPLED = 2 };

// First half: miss / hit data / alpha coin / emission / direction sampling (raytracer.h:555-571).
//   SHADE_END     path finished (radiance updated)
//   SHADE_PASS    alpha pass-through: continue from `o` (updated) along the same `d`
//   SHADE_SAMPLED a direction was sampled; call shade_finish with the light pdf of (mid.pos, mid.dir)
RT_HD ShadeStep shade_begin(const DScene &s, const float *lut, const RngKey &key, uint32_t bounce, bool last_bounce,
                            const Hit &h, f3 &o, const f3 &d, const f3 &thr, f3 &radiance, ShadeMid &mid) {
    if (h.tri < 0) {  // miss: Scene::bg_at, scene.h:83-89
        radiance = radiance + thr * bg_at(s, lut, d);
        return SHADE_END;
    }
    mid.sf = make_surface(s, lut, h, d);
    mid.pos = o + d * h.t;  // ray.at(t): the next ray starts exactly here, no normal offset
    const u4 r0 = rng_block(key, bounce, 0);
    if (!(u01(r0.x) <= mid.sf.alpha)) {  // alpha pass-through consumes a bounce, drops this hit's emission (raytracer.h:559-561)
        o = mid.pos;
        return last_bounce ? SHADE_END : SHADE_PASS;
    }
    radiance = radiance + thr * mid.sf.emission;  // every remaining exit of shade() returns emission (+ ...)
    if (last_bounce) return SHADE_END;            // trace_ray(depth 0) = 0, raytracer.h:596-598
    const float rough = fmaxf(mid.sf.roughness, s.min_roughness);
    mid.alpha = rough * rough;
    mid.nx = choose_local_x(mid.sf.ns);
    if (u01(r0.y) <= s.vndf_factor) {
        mid.dir = vndf_sample(mid.alpha, d, mid.sf.ns, mid.nx, u01(r0.z), u01(r0.w));
    } else {
        const u4 r1 = rng_block(key, bounce, 1);
        // mix_dist{cosine, bvh_mix}: uniform selector, raytracer.h:383-392; cosine only without lights (:449-453)
        const bool pick_light = s.n_lights > 0 && !(u01(r0.z) * 2.0f < 1.0f);
        mid.dir = pick_light ? light_sample(s, mid.pos, u01(r0.w), u01(r1.x), u01(r1.y))
                             : cosine_sample(mid.sf.ng, u01(r1.x), u01(r1.y));
    }
    if (any_nan(mid.dir)) return SHADE_END;  // raytracer.h:569-571
    return SHADE_SAMPLED;
}

// Second half: pdf mixture, BRDF, throughput (raytracer.h:572-590), in two steps so that the wavefront can
// obtain the light pdf of (mid.pos, mid.dir) from the traversal kernel between them:
//   shade_weights: everything that does not need the light pdf
//        f_cos     = pbr_brdf * max(0, dir . Ns)
//        p_partial = VNDF_factor * p_vndf + (1 - VNDF_factor) * p_cos * (1/2 with lights, 1 without)
//   shade_resolve: p = p_partial + (1 - VNDF_factor)/2 * p_light;  p < EPS -> the path ends (raytracer.h:576-578);
//        scl = f_cos / p;  |scl|^2 == 0 -> ends (raytracer.h:584-586);  thr *= scl.
// Same terms as the reference's `pbr_brdf * (max(0, cos) / p)` with p = 1/3 p_vndf + 2/3 (p_cos + p_light)/2, summed
// in a different order (differences of a few ulp).
struct ShadeWeights {
    f3 f_cos;
    float p_partial;
};
RT_HD ShadeWeights shade_weights(const DScene &s, const ShadeMid &mid, f3 d_in) {
    ShadeWeights w;
    const f3 h = normalize(mid.dir - d_in);  // halfway (raytracer.h:131-134): one IEEE normalisation for the pdf and the BRDF
    const float p_vndf = vndf_pdf(mid.alpha, s.eps, d_in, mid.sf.ns, mid.nx, h);
    const float p_cos = cosine_pdf(mid.sf.ng, mid.dir);
    const float k = s.n_lights > 0 ? 0.5f : 1.0f;  // mix_dist::pdf = mean of the sub-pdfs, raytracer.h:395-407
    w.p_partial = s.vndf_factor * p_vndf + (1.0f - s.vndf_factor) * k * p_cos;
    w.f_cos = pbr_brdf(mid.sf, mid.alpha, d_in, mid.dir, h) * fmaxf(0.0f, dot(mid.dir, mid.sf.ns));
    return w;
}
RT_HD float light_pdf_weight(const DScene &s) { return s.n_lights > 0 ? (1.0f - s.vndf_factor) * 0.5f : 0.0f; }

// thr_f = throughput * f_cos.  Returns false when the path ends; else thr = thr_f / p.
RT_HD bool shade_resolve(const DScene &s, f3 thr_f, float p_partial, float p_light, f3 &thr) {
    const float p = p_partial + light_pdf_weight(s) * p_light;
    if (p < s.eps) return false;  // NaN p continues, like the reference
    const f3 scaled = thr_f * sh_rcp(p);
    if (len2(scaled) == 0.0f) return false;
    thr = scaled;
    return true;
}

RT_HD bool shade_finish(const DScene &s, const ShadeMid &mid, float p_light, f3 &o, f3 &d, f3 &thr) {
    const ShadeWeights w = shade_weights(s, mid, d);
    if (len2(w.f_cos) == 0.0f) return false;  // raytracer.h:584-586 (decidable before the light pdf is known)
    if (!shade_resolve(s, thr * w.f_cos, w.p_partial, p_light, thr)) return false;
    o = mid.pos;
    d = mid.dir;
    return true;
}

RT_HD bool shade_bounce(const DScene &s, const float *lut, const RngKey &key, uint32_t bounce, bool last_bounce,
                        const Hit &h, f3 &o, f3 &d, f3 &thr, f3 &radiance, uint32_t &light_rays) {
    ShadeMid mid;
    const ShadeStep step = shade_begin(s, lut, key, bounce, last_bounce, h, o, d, thr, radiance, mid);
    if (step != SHADE_SAMPLED) return step == SHADE_PASS;
    float p_light = 0.0f;
    if (s.n_lights > 0) {
        p_light = light_pdf(s, mid.pos, mid.dir);
        ++light_rays;
    }
    return shade_finish(s, mid, p_light, o, d, thr);
}

// sanitize_nans, raytracer.h:607-616: per channel NaN -> 0, Inf kept
RT_HD f3 sanitize(f3 c) { return mk3(c.x != c.x ? 0.0f : c.x, c.y != c.y ? 0.0f : c.y, c.z != c.z ? 0.0f : c.z); }

}  // namespace rt

#endif  // RT_PT_CORE_CUH
