// aov.cuh — AOV render (rt_gpu_render_aov): per-pixel feature buffers from the camera samples of the beauty render.
//
// Every camera sample walks the beauty path's alpha pass-throughs with the beauty path's own coins and stops at its
// visible surface, whose make_surface values (base colour, shading normal, emission), distance along the camera ray
// and coverage 1 are the sample's values; a miss or ray_depth pass-throughs give zeros.  The wavefront is the beauty
// render's, with k_shade replaced:
//
//   k_generate / k_generate_views / k_generate_proj   queue 0, unchanged: the same camera rays bit for bit
//   for bounce b in [0, ray_depth):
//     k_extend (k_extend8)   closest hits of queue b, unchanged
//     k_aov_step             aov_visit per entry: the sample's values into its slot, or (pass-through) the ray into
//                            queue b + 1 with a warp-aggregated append
//   k_aov_accumulate         per-pixel float sums of the slots in k_accumulate's sample order
//
// Storage per path, beyond the beauty queues: three float4 slots, indexed like the radiance slot
// (sample - s0) * npix + (key - pix0), so that the order of the appends changes no bit:
//   a = (albedo.rgb, coverage), b = (normal.xyz, depth), c = (emission.rgb, 0)
// The per-pixel sums are the same three planes.  A pass-through ray carries the distance from the camera ray's origin
// to its own origin in thr.x; the rest of its record is emit_ray_record's (key in o.w, sample in d.w, not pending), so
// k_extend and k_extend8 read nothing else at b > 0 (the light pdf of a pending ray is never asked for).
//
// aov_visit is compiled for the host as well (tests/hostcheck/aovcheck.cpp: hc_aov).
#ifndef RT_AOV_CUH
#define RT_AOV_CUH

#include "pt_core.cuh"

namespace rt {

// The values of one camera sample: make_surface's at its visible surface, all zero when it has none
struct AovSample {
    f3 albedo, normal, emission;
    float depth, coverage;
};

// One hit h of the visible-surface walk of sample `key` at bounce b along the ray (o, d); depth_before = the distance
// from the camera ray's origin to o (0 at bounce 0).  Returns true when the sample passes through this hit with
// shade_begin's alpha coin and goes on: next_o = o + d * h.t (shade_begin's mid.pos), depth = depth_before + h.t.
// Otherwise `out` holds the sample's values: a miss, or a pass-through at the last bounce, gives zeros.
RT_HD bool aov_visit(const DScene &s, const float *lut, const RngKey &key, uint32_t bounce, bool last_bounce, const Hit &h, f3 o, f3 d,
                     float depth_before, AovSample &out, f3 &next_o, float &depth) {
    out.albedo = out.normal = out.emission = mk3(0.0f, 0.0f, 0.0f);
    out.depth = out.coverage = 0.0f;
    if (h.tri < 0) return false;
    const Surface sf = make_surface<1>(s, lut, h, d);  // its own out-of-line tex_sample (pt_core.cuh)
    const u4 r0 = rng_block(key, bounce, 0);
    if (!(u01(r0.x) <= sf.alpha)) {  // shade_begin's pass-through
        next_o = o + d * h.t;
        depth = depth_before + h.t;
        return !last_bounce;
    }
    out.albedo = sf.color;
    out.normal = sf.ns;
    out.emission = sf.emission;
    out.depth = depth_before + h.t;
    out.coverage = 1.0f;
    return false;
}

}  // namespace rt

#if defined(__CUDACC__)
#include "kernels.cuh"

namespace rt {

// Three float4 planes: per path slot (k_aov_step) or per pixel (k_aov_accumulate)
struct AovPlanes {
    float4 *a, *b, *c;  // (albedo.rgb, coverage), (normal.xyz, depth), (emission.rgb, 0)
};

constexpr int kAovThreads = 128;

// Bounce b of the AOV render: for every entry of queue b (hit by k_extend) aov_visit, then either the sample's values
// into its slot or the pass-through ray into queue b + 1.  bp is k_shade's (pix0 shifted by the views' key offset).
// A grid-stride loop over whole warps: the queue's size is read on the device.
__global__ void __launch_bounds__(kAovThreads) k_aov_step(DScene s, const float *__restrict__ lut_g, BatchParams bp, Queues q, uint32_t bounce,
                                                          AovPlanes slots) {
    __shared__ float lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = lut_g[i];
    __syncthreads();
    const uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t count = q.count[bounce * kCounterStride];
    uint32_t *const out_counter = q.count + (bounce + 1) * kCounterStride;
    const bool last = bounce + 1 == s.ray_depth;
    const uint32_t lane = lane_id();
    const uint32_t stride = gridDim.x * blockDim.x;
    uint32_t n_ext = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i - lane < count; i += stride) {  // warp-uniform condition
        bool pass = false;
        f3 o = mk3(0, 0, 0), d = mk3(0, 0, 1);
        float depth = 0.0f;
        uint32_t pixel = 0, sample = 0;
        if (i < count) {
            const float4 o4 = q.o_in[i], d4 = q.d_in[i], h4 = q.hit[i];
            const float depth_before = bounce ? q.thr_in[i].x : 0.0f;  // queue 0: camera rays
            o = mk3(o4.x, o4.y, o4.z);
            d = mk3(d4.x, d4.y, d4.z);
            pixel = __float_as_uint(o4.w);
            sample = __float_as_uint(d4.w) & 0x7FFFFFFFu;
            Hit h;
            h.t = h4.x;
            h.b = h4.y;
            h.c = h4.z;
            h.tri = __float_as_int(h4.w);
            const RngKey key{pixel, sample, bp.k0, bp.k1};
            AovSample v;
            f3 next_o = o;
            pass = aov_visit(s, lut, key, bounce, last, h, o, d, depth_before, v, next_o, depth);
            if (pass) {
                o = next_o;
            } else {
                const uint32_t slot = (sample - bp.s0) * bp.npix + (pixel - bp.pix0);
                slots.a[slot] = make_float4(v.albedo.x, v.albedo.y, v.albedo.z, v.coverage);
                slots.b[slot] = make_float4(v.normal.x, v.normal.y, v.normal.z, v.depth);
                slots.c[slot] = make_float4(v.emission.x, v.emission.y, v.emission.z, 0.0f);
            }
            ++n_ext;  // this extension ray's hit is consumed
        }
        const uint32_t mask = __ballot_sync(FULL, pass);
        uint32_t dst = 0;
        if (lane == 0 && mask) dst = atomicAdd(out_counter, static_cast<uint32_t>(__popc(mask)));
        dst = __shfl_sync(FULL, dst, 0) + static_cast<uint32_t>(__popc(mask & ((1u << lane) - 1u)));
        if (pass) {
            q.o_out[dst] = make_float4(o.x, o.y, o.z, __uint_as_float(pixel));
            q.d_out[dst] = make_float4(d.x, d.y, d.z, __uint_as_float(sample));
            q.thr_out[dst] = make_float4(depth, 1.0f, 1.0f, -1.0f);
        }
    }
    __shared__ uint32_t s_ext;
    if (threadIdx.x == 0) s_ext = 0;
    __syncthreads();
    for (int off = 16; off > 0; off >>= 1) n_ext += __shfl_down_sync(FULL, n_ext, off);
    if (lane == 0) atomicAdd(&s_ext, n_ext);
    __syncthreads();
    if (threadIdx.x == 0 && s_ext) atomicAdd(q.stats + 0, static_cast<unsigned long long>(s_ext));
}

__device__ __forceinline__ float4 sanitize4(float4 v) {
    return make_float4(v.x != v.x ? 0.0f : v.x, v.y != v.y ? 0.0f : v.y, v.z != v.z ? 0.0f : v.z, v.w != v.w ? 0.0f : v.w);
}

// sums[pixel] += sum_j sanitize(slot[j * npix + p]) for each plane: k_accumulate's NaN scrub, order and additions
__global__ void __launch_bounds__(256) k_aov_accumulate(BatchParams bp, AovPlanes slots, AovPlanes sums) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= bp.npix) return;
    float4 *const src[3] = {slots.a, slots.b, slots.c};
    float4 *const dst[3] = {sums.a, sums.b, sums.c};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float4 sum = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        for (uint32_t j = 0; j < bp.k; ++j) {
            const float4 v = sanitize4(src[k][static_cast<size_t>(j) * bp.npix + p]);
            sum.x = sum.x + v.x;
            sum.y = sum.y + v.y;
            sum.z = sum.z + v.z;
            sum.w = sum.w + v.w;
        }
        float4 a = dst[k][bp.pix0 + p];
        a.x += sum.x;
        a.y += sum.y;
        a.z += sum.z;
        a.w += sum.w;
        dst[k][bp.pix0 + p] = a;
    }
}

// rt_gpu_readback_aov: the means `sum / samples` (k_means' IEEE division) into one buffer of 11 * n floats:
// albedo [n * 3], normal [n * 3], emission [n * 3], depth [n], coverage [n]
__global__ void __launch_bounds__(256) k_aov_means(AovPlanes sums, float samples, uint32_t n, float *__restrict__ out) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const float4 a = sums.a[p], b = sums.b[p], c = sums.c[p];
    const size_t n3 = static_cast<size_t>(n) * 3, p3 = static_cast<size_t>(p) * 3;
    float *const albedo = out, *const normal = out + n3, *const emission = out + 2 * n3, *const depth = out + 3 * n3, *const coverage = depth + n;
    albedo[p3 + 0] = __fdiv_rn(a.x, samples);
    albedo[p3 + 1] = __fdiv_rn(a.y, samples);
    albedo[p3 + 2] = __fdiv_rn(a.z, samples);
    coverage[p] = __fdiv_rn(a.w, samples);
    normal[p3 + 0] = __fdiv_rn(b.x, samples);
    normal[p3 + 1] = __fdiv_rn(b.y, samples);
    normal[p3 + 2] = __fdiv_rn(b.z, samples);
    depth[p] = __fdiv_rn(b.w, samples);
    emission[p3 + 0] = __fdiv_rn(c.x, samples);
    emission[p3 + 1] = __fdiv_rn(c.y, samples);
    emission[p3 + 2] = __fdiv_rn(c.z, samples);
}

}  // namespace rt
#endif  // __CUDACC__

#endif  // RT_AOV_CUH
