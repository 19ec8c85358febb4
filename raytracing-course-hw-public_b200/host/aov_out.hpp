// aov_out.hpp — RT_AOV=<samples> of the reference-hosted CLI (main_ref_host.cpp): after the beauty render, the AOV
// render (rt_gpu_render_aov) of the scene camera, RT_PROJECTION honoured, with the same seed, written as portable float
// maps next to the image: <stem>_albedo.pfm, _normal, _emission, _depth and _coverage ("PF" for 3 channels, "Pf" for
// 1, little-endian scale -1, rows bottom to top), as the Python CLI writes them.  Needs only rt_gpu.h.
#ifndef RT_AOV_OUT_HPP
#define RT_AOV_OUT_HPP

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <stdexcept>
#include <string>
#include <vector>

#include "rt_gpu.h"

namespace rt_aov {

// RT_AOV's value -> samples (unset or empty: 0 = off); throws on anything but a non-negative integer
inline unsigned parse_samples(const char *v) {
    if (!v || !*v) return 0;
    for (const char *c = v; *c; ++c)
        if (*c < '0' || *c > '9')
            throw std::runtime_error(std::string("RT_AOV=") + v + ": expected the AOV render's samples per pixel, an integer >= 0");
    return static_cast<unsigned>(std::strtoul(v, nullptr, 10));
}

// w x h pixels of `channels` (1 or 3) floats, top row first, as a little-endian PFM
inline void write_pfm(const std::string &path, const float *data, unsigned w, unsigned h, int channels) {
    std::FILE *f = std::fopen(path.c_str(), "wb");
    if (!f) throw std::runtime_error("cannot write " + path);
    std::fprintf(f, "%s\n%u %u\n-1\n", channels == 3 ? "PF" : "Pf", w, h);
    const size_t row = static_cast<size_t>(w) * channels;
    for (unsigned y = h; y-- > 0;) std::fwrite(data + y * row, sizeof(float), row, f);  // x86: little-endian floats
    if (std::fclose(f) != 0) throw std::runtime_error("cannot write " + path);
}

// The AOV render of `samples` spp of `camera` (projection == nullptr: pinhole) on gpu, written next to out_path.
// gpu == nullptr (a scene of ray depth 0, which is not rendered): every buffer is 0.
inline void render_and_write(rt_gpu_ctx *gpu, unsigned width, unsigned height, unsigned samples, uint64_t seed, uint32_t max_paths,
                             const rt_camera *camera, const rt_projection *projection, const std::string &out_path) {
    const size_t n = static_cast<size_t>(width) * height;
    std::vector<float> albedo(n * 3, 0.0f), normal(n * 3, 0.0f), emission(n * 3, 0.0f), depth(n, 0.0f), coverage(n, 0.0f);
    if (gpu) {
        rt_render_params params{};
        params.width = width;
        params.height = height;
        params.samples = samples;
        params.mode = RT_MODE_BEAUTY;
        params.seed = seed;
        params.max_paths_in_flight = max_paths;
        const rt_views views{1, 0, camera};
        auto check = [](int rc, const char *what) {
            if (rc != RT_OK) throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + rt_gpu_last_error());
        };
        check(rt_gpu_render_aov(gpu, &params, projection ? &views : nullptr, projection), "rt_gpu_render_aov");
        rt_stats stats{};
        check(rt_gpu_readback_aov(gpu, albedo.data(), normal.data(), emission.data(), depth.data(), coverage.data(), &stats),
              "rt_gpu_readback_aov");
        std::fprintf(stderr, "rt_gpu AOV: %u spp, %.1f ms, %.1f Mrays/s (extension)\n", samples, stats.render_ms,
                     stats.extension_rays / (stats.render_ms > 0 ? stats.render_ms : 1e-9) * 1e-3);
    }
    const std::filesystem::path out(out_path);
    const std::string stem = (out.parent_path() / out.stem()).string();
    write_pfm(stem + "_albedo.pfm", albedo.data(), width, height, 3);
    write_pfm(stem + "_normal.pfm", normal.data(), width, height, 3);
    write_pfm(stem + "_emission.pfm", emission.data(), width, height, 3);
    write_pfm(stem + "_depth.pfm", depth.data(), width, height, 1);
    write_pfm(stem + "_coverage.pfm", coverage.data(), width, height, 1);
}

}  // namespace rt_aov

#endif  // RT_AOV_OUT_HPP
