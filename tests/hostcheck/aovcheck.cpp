// aovcheck.cpp — TEST-ONLY host statement of the AOV render (rt_gpu_render_aov), built as libaovcheck.so next to
// libhostcheck.so.  It is the host compilation of hostcheck.cpp (the same scene packing, camera and `trace`, so that
// hc_aov and hc_hitinfo trace the same hits bit for bit) plus one entry point, hc_aov, which walks the visible surface
// of every camera sample with aov_visit (csrc/aov.cuh), the function k_aov_step calls.  Nothing outside tests/ builds
// or loads it.
#include "hostcheck.cpp"

#include "aov.cuh"

extern "C" {

// Sequential statement of the AOV render (rt_gpu_render_aov): the camera rays of hc_render (centre != 0: the pixel
// centres of RT_MODE_PRIMARY_IDS, sample 0 only), the visible-surface walk of aov_visit through `trace`, the per-sample
// values NaN-scrubbed and summed in sample order, divided by samples.  out: w * h * 11 floats per pixel, albedo (3),
// normal (3), emission (3), depth, coverage.
int hc_aov(const rt_scene_desc *sc, uint32_t w, uint32_t h, uint32_t samples, uint64_t seed, int centre, float *out) {
    HostScene hs;
    if (int rc = build(sc, hs)) return rc;
    const Camera cam = make_camera(hs.d, w, h);
    const uint32_t n_s = centre ? 1u : samples;
    for (uint32_t pix = 0; pix < w * h; ++pix) {
        float sum[11] = {0};
        for (uint32_t s = 0; s < n_s; ++s) {
            const RngKey key{pix, s, (uint32_t)seed, (uint32_t)(seed >> 32)};
            float jx = 0.5f, jy = 0.5f;
            if (!centre) {
                const u4 j = rng_jitter(key);
                jx = u01(j.x);
                jy = u01(j.y);
            }
            f3 o = cam.pos;
            const f3 d = camera_dir(cam, (float)(pix % w) + jx, (float)(pix / w) + jy);
            float depth = 0.0f;
            AovSample v;
            v.albedo = v.normal = v.emission = mk3(0, 0, 0);
            v.depth = v.coverage = 0.0f;
            for (uint32_t b = 0; b < hs.d.ray_depth; ++b) {
                const Hit hit = trace(hs.d.scene, o, d, hs.d.eps);
                f3 next_o = o;
                float next_depth = depth;
                if (!aov_visit(hs.d, hs.p.gamma_lut, key, b, b + 1 == hs.d.ray_depth, hit, o, d, depth, v, next_o, next_depth)) break;
                o = next_o;
                depth = next_depth;
            }
            const f3 a = sanitize(v.albedo), n = sanitize(v.normal), e = sanitize(v.emission);
            const float vals[11] = {a.x, a.y, a.z, n.x, n.y, n.z, e.x, e.y, e.z, v.depth != v.depth ? 0.0f : v.depth, v.coverage};
            for (int k = 0; k < 11; ++k) sum[k] = sum[k] + vals[k];
        }
        for (int k = 0; k < 11; ++k) out[(size_t)pix * 11 + k] = sum[k] / (float)n_s;
    }
    return 0;
}

}  // extern "C"
