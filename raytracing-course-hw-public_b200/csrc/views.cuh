// views.cuh — multi-view rendering (rt_gpu_render_views): V cameras over one uploaded scene in one render.
//
// The V views of W x H are stacked into one image of W x (V * H) pixels: stacked pixel v * W * H + y * W + x is pixel
// (x, y) of view v.  Only queue 0 knows about views: k_generate_views splits the stacked pixel into (view, x, y) and
// reads that view's camera.  Its paths carry the Philox pixel key (view_base + v) * W * H + y * W + x, and the host
// hands k_shade a BatchParams whose pix0 is shifted by the same view_base * W * H, so k_shade's radiance slot
// (sample - s0) * npix + (pixel - pix0) is the one of the stacked render.  k_extend, k_shade, k_lightpdf_list,
// k_accumulate, the reduce and the readback kernels work on the stacked index unchanged.  The adaptive form
// (rt_gpu_render_views_adaptive) is the same with k_generate_active_views in place of k_generate_active; the rounds,
// the rule kernels and k_accumulate_active of adaptive.cuh work on the stacked index unchanged as well.
//
// The split is a pure function, compiled for the host as well (tests).
#ifndef RT_VIEWS_CUH
#define RT_VIEWS_CUH

#include <stdint.h>

#if defined(__CUDACC__)
#define RT_VIEWS_HD __host__ __device__ __forceinline__
#else
#define RT_VIEWS_HD inline
#endif

namespace rt {

struct ViewPixel {
    uint32_t view, x, y;
};

// Stacked pixel -> (view, x, y) of views of width x height (width * height < 2^31, checked on the host)
RT_VIEWS_HD ViewPixel split_view_pixel(uint32_t pixel, uint32_t width, uint32_t height) {
    const uint32_t per_view = width * height;
    const uint32_t view = pixel / per_view;
    const uint32_t local = pixel - view * per_view;
    const uint32_t y = local / width;
    return ViewPixel{view, local - y * width, y};
}

}  // namespace rt

#if defined(__CUDACC__)
#include "kernels.cuh"

namespace rt {

// Queue 0 of a multi-view batch: k_generate over the stacked image, with the camera of each path's view.  The slot,
// tile and radiance-slot rules are k_generate's; bp is the stacked batch (pix0 a stacked index, height the height of
// one view) and key_offset = view_base * W * H turns a stacked pixel into its Philox pixel key.  With W % 8 == 0 and
// H % 4 == 0 an 8 x 4 tile lies in one view, so a warp reads one camera.
__global__ void __launch_bounds__(256) k_generate_views(const Camera *__restrict__ cams, BatchParams bp, Queues q, uint32_t key_offset) {
    const uint32_t n = bp.npix * bp.k;
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot == 0) {
        q.count[0] = n;
        atomicAdd(q.stats + 3, static_cast<unsigned long long>(n));
    }
    if (slot >= n) return;
    const uint32_t j = slot / bp.npix;
    const uint32_t pl = slot - j * bp.npix;
    const uint32_t pixel = bp.tiled ? tiled_pixel(pl, bp.width) : bp.pix0 + pl;
    const ViewPixel vp = split_view_pixel(pixel, bp.width, bp.height);
    emit_camera_ray_at(cams[vp.view], bp, q, slot, slot, pixel + key_offset, vp.x, vp.y, bp.s0 + j);
}

// Queue 0 of an adaptive multi-view batch (rt_gpu_render_views_adaptive): k_generate_active (adaptive.cuh) over the
// stacked image.  The list holds stacked pixels; bp is the unshifted stacked batch (pix0 / npix = the whole range,
// height the height of one view), so the radiance slot j * npix + (pixel - pix0) is the one k_shade derives from the
// key pixel + key_offset with its pix0 shifted by the same key_offset.
__global__ void __launch_bounds__(256) k_generate_active_views(const Camera *__restrict__ cams, BatchParams bp, Queues q,
                                                               const uint32_t *__restrict__ list, const uint32_t *__restrict__ active,
                                                               uint32_t key_offset) {
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
    const ViewPixel vp = split_view_pixel(pixel, bp.width, bp.height);
    emit_camera_ray_at(cams[vp.view], bp, q, slot, j * bp.npix + (pixel - bp.pix0), pixel + key_offset, vp.x, vp.y, bp.s0 + j);
}

}  // namespace rt
#endif  // __CUDACC__

#endif  // RT_VIEWS_CUH
