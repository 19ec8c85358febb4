// adaptive.cuh — adaptive sampling (rt_gpu_render_adaptive): every pixel of the range traces samples in rounds until
// its relative noise reaches a target or it reaches the maximum spp.
//
//   round 0        every pixel of [pixel_begin, pixel_end) gets min_samples samples
//   round r > 0    every pixel still on the ACTIVE LIST gets step_samples more (the last round clipped at the maximum)
//   per round      ceil(k / k_max) batches of  k_generate_active -> bounces (k_extend / k_shade / k_lightpdf_list, the
//                  fixed render's kernels, untouched) -> k_accumulate_active;  then k_adapt_flags (the rule, one bit per
//                  list entry) -> rtb::kb_scan (gpu_build.cuh) -> k_adapt_scatter (stable compaction into the other list)
//
// A pixel always receives the sample prefix [0, n_p), and Philox is keyed by (pixel, sample), so an adaptive image is,
// pixel by pixel, a fixed render truncated at that pixel's count.  A batch keeps bp.pix0 / bp.npix equal to the whole
// rendered range, so k_shade's radiance slot (sample - s0) * npix + (pixel - pix0) stays what it is in a fixed render;
// only queue 0 is sparse (n_active * k paths).  Every size is read on the device: the host never waits for a round.
//
// Per pixel, accum = (sum r, sum g, sum b, Q = sum y^2) with y = (r + g + b) / 3 of each sanitised sample, counts = n.
// The stopping rule (adapt_rel_error) is a pure function, compiled for the host as well (tests).
#ifndef RT_ADAPTIVE_CUH
#define RT_ADAPTIVE_CUH

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define RT_ADAPT_HD __host__ __device__ __forceinline__
#else
#define RT_ADAPT_HD inline
#endif

namespace rt {

// Relative standard error of a pixel's mean luminance from S = sum y, Q = sum y^2 over n >= 2 samples (double):
//   m = S / n,  var = max(Q / n - m^2, 0) * n / (n - 1),  err = sqrt(var / n) / (m + abs_floor)
// abs_floor > 0 keeps near-black pixels from chasing relative noise.
RT_ADAPT_HD double adapt_rel_error(double S, double Q, uint32_t n, double abs_floor) {
    if (n < 2) return INFINITY;
    const double nd = static_cast<double>(n);
    const double m = S / nd;
    const double var = fmax(Q / nd - m * m, 0.0) * nd / (nd - 1.0);
    return sqrt(var / nd) / (m + abs_floor);
}

// S of a pixel from its rgb sums
RT_ADAPT_HD double adapt_luma_sum(float r, float g, float b) {
    return (static_cast<double>(r) + static_cast<double>(g) + static_cast<double>(b)) / 3.0;
}

// A pixel stops once err <= rel_error; rel_error == 0 never stops early.  NaN (an infinite sample) never stops.
RT_ADAPT_HD bool adapt_converged(double err, float rel_error) { return rel_error > 0.0f && err <= static_cast<double>(rel_error); }

}  // namespace rt

#if defined(__CUDACC__)
#include "gpu_build.cuh"
#include "kernels.cuh"

namespace rt {

// The first active list: the range's pixels in k_generate's 8 x 4 tile order when the batch is the whole image and
// the image is made of whole tiles (tiled != 0), else row-major.  active[0] = the list's length.
__global__ void __launch_bounds__(256) k_adapt_init(uint32_t *__restrict__ list, uint32_t pix0, uint32_t n_render, uint32_t width,
                                                    uint32_t tiled, uint32_t *__restrict__ active) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) active[0] = n_render;
    if (i >= n_render) return;
    list[i] = tiled ? tiled_pixel(i, width) : pix0 + i;
}

// Queue 0 of an adaptive batch: n_active * k camera rays, slot = j * n_active + list position.  The grid covers the
// whole range (npix * k); the threads past the device-side count exit.
__global__ void __launch_bounds__(256) k_generate_active(Camera cam, BatchParams bp, Queues q, const uint32_t *__restrict__ list,
                                                         const uint32_t *__restrict__ active) {
    const uint32_t n_act = *active;
    const uint32_t n = n_act * bp.k;
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot == 0) {
        q.count[0] = n;
        atomicAdd(q.stats + 3, static_cast<unsigned long long>(n));
    }
    if (slot >= n) return;
    const uint32_t j = slot / n_act;
    const uint32_t li = slot - j * n_act;
    const uint32_t pixel = list[li];
    emit_camera_ray(cam, bp, q, slot, j * bp.npix + (pixel - bp.pix0), pixel, bp.s0 + j);
}

// accum[pixel] += (rgb sums in k_accumulate's order, sum of y^2); counts[pixel] += k — one thread per list entry
__global__ void __launch_bounds__(256) k_accumulate_active(BatchParams bp, const float4 *__restrict__ rad, float4 *__restrict__ accum,
                                                           uint32_t *__restrict__ counts, const uint32_t *__restrict__ list,
                                                           const uint32_t *__restrict__ active) {
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= *active) return;
    const uint32_t pixel = list[li];
    const float4 sum = sum_samples<true>(bp, rad, pixel - bp.pix0);
    float4 a = accum[pixel];
    a.x += sum.x;
    a.y += sum.y;
    a.z += sum.z;
    a.w += sum.w;
    accum[pixel] = a;
    counts[pixel] += bp.k;
}

// The rule for every list entry: err map, and one bit per entry that goes on (words[li / 32], ballot).  The grid
// covers n_words * 32 entries so that the words past the device-side count are written as 0.
__global__ void __launch_bounds__(256) k_adapt_flags(const uint32_t *__restrict__ list, const uint32_t *__restrict__ active,
                                                     const float4 *__restrict__ accum, const uint32_t *__restrict__ counts,
                                                     float *__restrict__ err, uint32_t max_samples, float rel_error, float abs_floor,
                                                     uint32_t *__restrict__ words, uint32_t n_words) {
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    bool more = false;
    if (li < *active) {
        const uint32_t pixel = list[li];
        const float4 a = accum[pixel];
        const uint32_t n = counts[pixel];
        const double e = adapt_rel_error(adapt_luma_sum(a.x, a.y, a.z), static_cast<double>(a.w), n, static_cast<double>(abs_floor));
        err[pixel] = static_cast<float>(e);
        more = n < max_samples && !adapt_converged(e, rel_error);
    }
    const uint32_t w = __ballot_sync(0xFFFFFFFFu, more);
    if ((threadIdx.x & 31u) == 0 && (li >> 5) < n_words) words[li >> 5] = w;
}

// Stable compaction of the entries whose bit is set into the other list (wscan = rtb::kb_scan of the words, whose total
// is the next round's active count)
__global__ void __launch_bounds__(256) k_adapt_scatter(const uint32_t *__restrict__ list, uint32_t *__restrict__ next,
                                                       const uint32_t *__restrict__ active, const uint32_t *__restrict__ words,
                                                       const uint32_t *__restrict__ wscan) {
    const uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= *active) return;
    const uint32_t w = words[li >> 5], bit = 1u << (li & 31u);
    if (w & bit) next[wscan[li >> 5] + __popc(w & (bit - 1u))] = list[li];
}

// rt_gpu_readback after an adaptive render: per-pixel means sum / n (IEEE division, like k_means); 0 where n == 0
__global__ void __launch_bounds__(256) k_means_counts(const float4 *__restrict__ accum, const uint32_t *__restrict__ counts,
                                                      uint32_t n_pixels, float *__restrict__ rgb) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const float4 a = accum[p];
    const uint32_t n = counts[p];
    const float s = static_cast<float>(n);
    rgb[static_cast<size_t>(p) * 3 + 0] = n ? __fdiv_rn(a.x, s) : 0.0f;
    rgb[static_cast<size_t>(p) * 3 + 1] = n ? __fdiv_rn(a.y, s) : 0.0f;
    rgb[static_cast<size_t>(p) * 3 + 2] = n ? __fdiv_rn(a.z, s) : 0.0f;
}

// rt_gpu_readback_rgb8 after an adaptive render: k_tonemap of the same means (pixels without samples -> 0)
__global__ void __launch_bounds__(256) k_tonemap_counts(const float4 *__restrict__ accum, const uint32_t *__restrict__ counts,
                                                        uint32_t n_pixels, uint8_t *__restrict__ rgb8) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pixels) return;
    const uint32_t n = counts[p];
    uint8_t *out = rgb8 + static_cast<size_t>(p) * 3;
    if (n) {
        tonemap_pixel(accum[p], static_cast<float>(n), out);
    } else {
        out[0] = out[1] = out[2] = 0;
    }
}

}  // namespace rt
#endif  // __CUDACC__

#endif  // RT_ADAPTIVE_CUH
