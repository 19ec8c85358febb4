// projection.cuh — camera projections (rt_gpu_render_projected): pinhole, thin lens, orthographic and equirectangular
// views over the 64-byte rt::Camera (position and basis) of a multi-view render.
//
// Only queue 0 knows about projections.  k_generate_proj / k_generate_active_proj are k_generate_views /
// k_generate_active_views (views.cuh) with a per-view Projection next to the camera: same slots, tile order, Philox
// pixel key (pixel + view_base * W * H) and radiance slots.  k_extend, k_shade, k_lightpdf_list and k_accumulate* see a
// ray origin, a direction and a key, as for any camera ray.
//
// Random numbers: the pixel jitter is rng_jitter (counter word 2 = 0xFFFFFFFF, lanes 0-1) as in every render; the lens
// sample of a thin lens with a non-zero aperture is rng_lens (counter word 2 = 0xFFFFFFFE, lanes 0-1), drawn only for
// such a view.  A pinhole view draws exactly what k_generate draws.  Pixel-centre rays (RT_MODE_PRIMARY_IDS) use the
// pixel centre and the lens centre, i.e. the pinhole ray for a thin lens.
//
// projected_ray is a pure function, compiled for the host as well (tests).
#ifndef RT_PROJECTION_CUH
#define RT_PROJECTION_CUH

#include "pt_core.cuh"

namespace rt {

// Values of Projection::kind; equal to RT_PROJ_* of rt_gpu.h
constexpr uint32_t kProjPinhole = 0, kProjThinLens = 1, kProjOrthographic = 2, kProjEquirect = 3;

// Same layout as rt_projection (rt_gpu.h).  Fields a kind does not use are ignored.
struct Projection {
    uint32_t kind;
    float aperture_radius, focus_distance;  // thin lens: lens radius and the distance of the plane in focus along fwd
    float half_width, half_height;          // orthographic: half the extent of the view along right / up (glTF xmag / ymag)
};

struct ProjectedRay {
    f3 o, d;
};

// Lens sample of a thin-lens path: counter word 2 = 0xFFFFFFFE, lanes 0 and 1
RT_HD u4 rng_lens(const RngKey &k) { return philox4x32_10(k.pixel, k.sample, 0xFFFFFFFEu, 0u, k.k0, k.k1); }

// Shirley and Chiu's concentric map of the unit square onto the unit disc (area-preserving, so uniform samples stay
// uniform).  (0.5, 0.5) maps to (0, 0) exactly.
RT_HD void concentric_disc(float lu, float lv, float &x, float &y) {
    const float a = 2.0f * lu - 1.0f, b = 2.0f * lv - 1.0f;
    if (a == 0.0f && b == 0.0f) {
        x = y = 0.0f;
        return;
    }
    float r, phi;
    if (fabsf(a) > fabsf(b)) {
        r = a;
        phi = (RT_PI * 0.25f) * (b / a);
    } else {
        r = b;
        phi = RT_PI * 0.5f - (RT_PI * 0.25f) * (a / b);
    }
    x = r * cosf(phi);
    y = r * sinf(phi);
}

// v, or +-2^-80 for a zero.  The node tests form (plane - o) * (1 / d); for d == 0 that is inf - inf = NaN, fmaxf /
// fminf drop it, and the slab of that axis stops culling: a ray with two zero components visits every node along the
// third axis.  A camera ray almost never has a zero component, but every ray of an orthographic view of an axis-aligned
// camera does.  2^-80 turns the axis into a finite slab test (1 / 2^-80 = 2^80, far from overflow for scene-sized
// distances) and moves the ray by nothing a float32 hit point can show.
RT_HD float nonzero(float v) { return v == 0.0f ? copysignf(0x1p-80f, v) : v; }

// The ray through image point (px, py) (pixel units, pixel centres at + 0.5) of camera c under projection p, with lens
// sample (lu, lv) in [0, 1)^2 (thin lens only):
//   pinhole          pos, camera_dir(c, px, py)
//   thin lens        d = camera_dir(c, px, py), focus = pos + d * (focus_distance / dot(d, fwd)),
//                    lens = pos + x * right + y * up with (x, y) = aperture_radius * concentric_disc(lu, lv),
//                    direction normalize(focus - lens); the pinhole ray when the lens point is the centre (aperture 0,
//                    or the lens centre (0.5, 0.5))
//   orthographic     a = (px * inv_w2 - 1) * half_width, b = (py * inv_h2 - 1) * half_height (camera_dir's signs),
//                    origin pos + a * right - b * up, direction normalize(fwd) with zero components made nonzero
//   equirectangular  u = (px - 0.5) / W, v = (py - 0.5) / H, phi = (u - 0.5) * 2 pi, theta = (0.5 - v) * pi,
//                    d = normalize(cos(theta) sin(phi) * right + sin(theta) * up + cos(theta) cos(phi) * fwd)
// The equirectangular half-pixel shift is bg_at's convention: tex_sample puts texel i of a map of width W at
// u = i / W, so with fwd = +x, right = +z, up = +y (the basis in which bg_at's map centre lies straight ahead) the
// centre of pixel (i, j) of a W x H view looks up texel (i, j) of a W x H environment map.
RT_HD ProjectedRay projected_ray(const Camera &c, const Projection &p, float px, float py, float lu, float lv) {
    if (p.kind == kProjOrthographic) {
        const float a = (px * c.inv_w2 - 1.0f) * p.half_width;
        const float b = (py * c.inv_h2 - 1.0f) * p.half_height;
        const f3 d = normalize(c.fwd);
        return ProjectedRay{c.pos + a * c.right - b * c.up, mk3(nonzero(d.x), nonzero(d.y), nonzero(d.z))};
    }
    if (p.kind == kProjEquirect) {
        const float u = (px - 0.5f) * (0.5f * c.inv_w2), v = (py - 0.5f) * (0.5f * c.inv_h2);
        const float phi = (u - 0.5f) * (2.0f * RT_PI), theta = (0.5f - v) * RT_PI;
        const float ct = cosf(theta);
        return ProjectedRay{c.pos, normalize((ct * sinf(phi)) * c.right + sinf(theta) * c.up + (ct * cosf(phi)) * c.fwd)};
    }
    const f3 d = camera_dir(c, px, py);
    if (p.kind != kProjThinLens || p.aperture_radius == 0.0f) return ProjectedRay{c.pos, d};
    float x, y;
    concentric_disc(lu, lv, x, y);
    if (x == 0.0f && y == 0.0f) return ProjectedRay{c.pos, d};
    const f3 focus = c.pos + d * (p.focus_distance / dot(d, c.fwd));
    const f3 lens = c.pos + (p.aperture_radius * x) * c.right + (p.aperture_radius * y) * c.up;
    return ProjectedRay{lens, normalize(focus - lens)};
}

}  // namespace rt

#if defined(__CUDACC__)
#include "kernels.cuh"
#include "views.cuh"

namespace rt {

// The projected camera ray through pixel (px, py) of view (cam, pj) for Philox key (pixel, sample) into queue position
// `slot`, its radiance slot `rad_slot` cleared (emit_camera_ray_at with projected_ray in place of camera_dir)
__device__ __forceinline__ void emit_projected_ray_at(const Camera &cam, const Projection &pj, const BatchParams &bp, const Queues &q,
                                                      uint32_t slot, uint32_t rad_slot, uint32_t pixel, uint32_t px, uint32_t py,
                                                      uint32_t sample) {
    const RngKey key{pixel, sample, bp.k0, bp.k1};
    float jx = 0.5f, jy = 0.5f, lu = 0.5f, lv = 0.5f;
    if (!bp.centre) {
        const u4 r = rng_jitter(key);
        jx = u01(r.x);
        jy = u01(r.y);
        if (pj.kind == kProjThinLens && pj.aperture_radius != 0.0f) {
            const u4 l = rng_lens(key);
            lu = u01(l.x);
            lv = u01(l.y);
        }
    }
    const ProjectedRay ray = projected_ray(cam, pj, static_cast<float>(px) + jx, static_cast<float>(py) + jy, lu, lv);
    emit_ray_record(bp, q, slot, rad_slot, pixel, sample, ray.o, ray.d);
}

// Queue 0 of a projected multi-view batch: k_generate_views with the projection of each path's view
__global__ void __launch_bounds__(256) k_generate_proj(const Camera *__restrict__ cams, const Projection *__restrict__ projs, BatchParams bp,
                                                       Queues q, uint32_t key_offset) {
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
    emit_projected_ray_at(cams[vp.view], projs[vp.view], bp, q, slot, slot, pixel + key_offset, vp.x, vp.y, bp.s0 + j);
}

// Queue 0 of an adaptive projected multi-view batch: k_generate_active_views with the projection of each path's view
__global__ void __launch_bounds__(256) k_generate_active_proj(const Camera *__restrict__ cams, const Projection *__restrict__ projs,
                                                              BatchParams bp, Queues q, const uint32_t *__restrict__ list,
                                                              const uint32_t *__restrict__ active, uint32_t key_offset) {
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
    emit_projected_ray_at(cams[vp.view], projs[vp.view], bp, q, slot, j * bp.npix + (pixel - bp.pix0), pixel + key_offset, vp.x, vp.y,
                          bp.s0 + j);
}

}  // namespace rt
#endif  // __CUDACC__

#endif  // RT_PROJECTION_CUH
