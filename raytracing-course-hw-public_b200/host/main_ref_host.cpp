// main_ref_host.cpp — the reference-hosted drop-in: `raytracer_b200 <scene.gltf|scene.txt> <width> <height> <samples> <out.ppm>`.
//
// Same five positional arguments, same exit codes and the same output file as the reference CLI
// (src/main.cpp:16-49).  Everything on the host is the reference's own code, used through its headers
// (-I<reference>/src, never copied): parse_gltf_scene (scene.h:183), the light-BVH build of
// RaytracerStaticContext (raytracer.h:444-447), Image::set_pixel's tonemap / gamma / quantisation
// (image.h:40-82) and Image::write (image.h:34).  The only replaced call is run_raytracer(scene, img)
// (main.cpp:37): the per-pixel Monte-Carlo loop runs on the B200(s) through the rt_gpu C ABI.
//
// A `*.txt` scene (the course's sample_data/scene-NNN.txt and homebrew_primitives/*.txt, which the reference at HEAD
// aborts on: main.cpp:27 calls the glTF loader unconditionally) goes through rt_text_scene_parse (librt_host) and
// rt_gpu_upload_text_scene; width / height / samples of 0 take the file's DIMENSIONS / SAMPLES.  PARITY UNPINNED
// (include/rt_gpu.h): no reference code exists for these scenes; the tonemap and the PPM writer are still the reference's.
//
// Optional environment (additions; the 5-argument form needs none of them):
//   RT_GPUS   number of GPUs of this box to split the samples over (default 1)
//   RT_SEED   Philox seed (default 0)
//   RT_PATHS  paths in flight per batch (default 128 Mi; the library's own default is 512 Mi)
//   RT_TIMING 1: wall time of the host phases on stderr
//   RT_HOST_SCENE_BVH  1: also build the reference's scene BVH and pass it (default: the library builds its own)
//   RT_ADD_LIGHT_TRIANGLE  1: the extra light source of the reference's compile-time ADD_LIGHT_TRIANGLE (config.h:39-47)
//   RT_ENV_MAP  image file used as the equirectangular environment map Scene::bg (the run-time form of the
//             reference's compile-time USE_ENV_MAP / ENV_MAP_PATH, src/config.h:35-37)
//   RT_ADAPTIVE  relative-error target of an adaptive render (rt_gpu_render_adaptive, glTF scenes): <samples> becomes
//             the maximum spp, min_samples = step_samples = max(2, ceil(samples / 16)); the samples traced on stderr
//   RT_PROJECTION  projection of the scene camera (rt_gpu_render_projected, glTF scenes): thin_lens:<aperture>:<focus>,
//             ortho:<half_w>:<half_h>, equirect or pinhole; combines with RT_ADAPTIVE
//   RT_AOV    samples per pixel of an AOV render after the beauty render (rt_gpu_render_aov, glTF scenes; same camera,
//             RT_PROJECTION and seed): <stem>_albedo.pfm, _normal, _emission, _depth and _coverage (aov_out.hpp)
#define STB_IMAGE_IMPLEMENTATION

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <fstream>
#include <iostream>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "config.h"
#include "geometry.h"
#include "image.h"
#include "raytracer.h"
#include "scene.h"

#include "aov_out.hpp"
#include "flatten_ref.hpp"
#include "rt_gpu.h"
#include "rt_host.h"

namespace {
void check(int rc, const char *what) {
    if (rc != RT_OK) throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + rt_gpu_last_error());
}
// RT_TIMING=1: wall time of the host phases on stderr
struct PhaseClock {
    bool on = std::getenv("RT_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char *what) {
        const auto n = std::chrono::steady_clock::now();
        if (on) std::fprintf(stderr, "raytracer_b200: %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};
unsigned env_uint(const char *name, unsigned fallback) {
    const char *v = std::getenv(name);
    return v && *v ? static_cast<unsigned>(std::strtoul(v, nullptr, 10)) : fallback;
}

// RT_PROJECTION's value -> p; false when it is malformed
bool parse_projection(const std::string &v, rt_projection &p) {
    p = rt_projection{};
    const size_t c1 = v.find(':'), c2 = c1 == std::string::npos ? c1 : v.find(':', c1 + 1);
    const std::string name = v.substr(0, c1);
    if (name == "pinhole" || name == "equirect") {
        p.kind = name == "pinhole" ? RT_PROJ_PINHOLE : RT_PROJ_EQUIRECT;
        return c1 == std::string::npos;
    }
    if ((name != "thin_lens" && name != "ortho") || c2 == std::string::npos || v.find(':', c2 + 1) != std::string::npos) return false;
    char *end1 = nullptr, *end2 = nullptr;
    const std::string a = v.substr(c1 + 1, c2 - c1 - 1), b = v.substr(c2 + 1);
    const float x = std::strtof(a.c_str(), &end1), y = std::strtof(b.c_str(), &end2);
    if (a.empty() || b.empty() || *end1 || *end2) return false;
    if (name == "thin_lens") {
        p.kind = RT_PROJ_THIN_LENS;
        p.aperture_radius = x;
        p.focus_distance = y;
    } else {
        p.kind = RT_PROJ_ORTHOGRAPHIC;
        p.half_width = x;
        p.half_height = y;
    }
    return true;
}

// render what was uploaded and feed the float means to the reference's Image::set_pixel (image.h:40).  camera: the
// scene camera that RT_PROJECTION applies to (nullptr: text scene, where it is refused).
void render_into(rt_gpu_ctx *gpu, unsigned width, unsigned height, unsigned samples, Image &img, const rt_camera *camera) {
    rt_render_params params{};
    params.width = width;
    params.height = height;
    params.samples = samples;
    params.mode = RT_MODE_BEAUTY;
    params.seed = env_uint("RT_SEED", 0);
    // A one-shot command pays for allocating and freeing the path queues: 128 Mi paths per batch (17 GB) instead of the
    // library's 512 Mi (68 GB) cost 1.7 % of the render and save ~0.15 s of cudaMalloc / cudaFree (RT_PATHS overrides).
    params.max_paths_in_flight = env_uint("RT_PATHS", 128u << 20);
    const char *adaptive = std::getenv("RT_ADAPTIVE");
    rt_adaptive_params ap{};
    ap.min_samples = ap.step_samples = std::max(2u, (samples + 15) / 16);
    ap.rel_error = adaptive && *adaptive ? std::strtof(adaptive, nullptr) : 0.0f;
    ap.abs_floor = 1e-3f;
    const char *projection = std::getenv("RT_PROJECTION");
    if (projection && *projection) {
        rt_projection proj;
        if (!camera) throw std::runtime_error("RT_PROJECTION applies to glTF scenes only");
        if (!parse_projection(projection, proj))
            throw std::runtime_error(std::string("RT_PROJECTION=") + projection +
                                     ": expected thin_lens:<aperture>:<focus>, ortho:<half_w>:<half_h>, equirect or pinhole");
        const rt_views views{1, 0, camera};
        check(rt_gpu_render_projected(gpu, &params, &views, &proj, adaptive && *adaptive ? &ap : nullptr), "rt_gpu_render_projected");
    } else if (adaptive && *adaptive) {
        check(rt_gpu_render_adaptive(gpu, &params, &ap), "rt_gpu_render_adaptive");
    } else {
        check(rt_gpu_render(gpu, &params), "rt_gpu_render");
    }
    std::vector<float> mean(static_cast<size_t>(width) * height * 3);
    rt_stats stats{};
    check(rt_gpu_readback(gpu, mean.data(), nullptr, &stats), "rt_gpu_readback");
    for (size_t i = 0; i < static_cast<size_t>(width) * height; ++i)
        img.set_pixel(static_cast<int>(i), {mean[i * 3], mean[i * 3 + 1], mean[i * 3 + 2]});
    std::fprintf(stderr, "rt_gpu: %.1f ms, %.1f Msamples/s, %.1f Mrays/s (extension) + %.1f Mrays/s (light pdf)\n", stats.render_ms,
                 stats.samples / stats.render_ms * 1e-3, stats.extension_rays / stats.render_ms * 1e-3,
                 stats.light_pdf_rays / stats.render_ms * 1e-3);
    if (adaptive && *adaptive) {
        const double full = static_cast<double>(width) * height * samples;
        std::fprintf(stderr, "rt_gpu adaptive (rel_error %s): %llu samples traced, %.3f of %.0f\n", adaptive,
                     static_cast<unsigned long long>(stats.samples), stats.samples / full, full);
    }
}

void write_image(Image &img, const char *path) {
    std::filesystem::path out_path = path;
    std::filesystem::create_directories(out_path.parent_path());
    std::ofstream out(out_path, std::ios::binary);
    img.write(out);
}

// course text scene: parser in librt_host, megakernel behind rt_gpu_upload_text_scene
int run_text_scene(const char *path, unsigned width, unsigned height, unsigned samples, const char *out_path) {
    if (rt_aov::parse_samples(std::getenv("RT_AOV"))) throw std::runtime_error("RT_AOV applies to glTF scenes only");
    rt_text_scene *ts = nullptr;
    if (int rc = rt_text_scene_parse(path, &ts))
        throw std::runtime_error(std::string("cannot parse text scene ") + path + " (" + std::to_string(rc) + ")");
    width = width ? width : ts->width;
    height = height ? height : ts->height;
    samples = samples ? samples : ts->samples;
    Image img(width, height, {ts->bg_color[0], ts->bg_color[1], ts->bg_color[2]});
    if (ts->ray_depth != 0 || ts->shading == RT_SHADE_FLAT) {
        rt_gpu_ctx *gpu = nullptr;
        check(rt_gpu_create(&gpu, static_cast<int>(env_uint("RT_GPUS", 1)), 0), "rt_gpu_create");
        check(rt_gpu_upload_text_scene(gpu, ts), "rt_gpu_upload_text_scene");
        render_into(gpu, width, height, samples, img, nullptr);
        rt_gpu_destroy(gpu);
    }
    rt_text_scene_free(ts);
    write_image(img, out_path);
    return EXIT_SUCCESS;
}
}  // namespace

int main(int argc, char **argv) try {
    if (argc < 6) {
        std::cerr << "Too few arguments: expected 6, got " << argc - 1 << std::endl;
        return EXIT_FAILURE;
    }
    const unsigned width = std::strtol(argv[2], nullptr, 10);
    const unsigned height = std::strtol(argv[3], nullptr, 10);
    const unsigned samples = std::strtol(argv[4], nullptr, 10);

    if (std::filesystem::path(argv[1]).extension() == ".txt") return run_text_scene(argv[1], width, height, samples, argv[5]);

    const unsigned aov_samples = rt_aov::parse_samples(std::getenv("RT_AOV"));  // refused before any work when malformed
    PhaseClock clock;
    Scene scene = parse_gltf_scene(std::filesystem::path(argv[1]), static_cast<float>(width) / height);
    clock.lap("parse_gltf_scene");
    scene.bg_color = {ENV_MAP_INTENSITY, ENV_MAP_INTENSITY, ENV_MAP_INTENSITY};
    if constexpr (USE_ENV_MAP) scene.bg = geometry::Texture::load_img(ENV_MAP_PATH);  // main.cpp:29-31
    if (const char *env = std::getenv("RT_ENV_MAP")) scene.bg = geometry::Texture::load_img(env);
    if (env_uint("RT_ADD_LIGHT_TRIANGLE", 0)) rt_flatten::append_light_triangle(scene);  // config.h:39-47 at run time
    scene.camera.width = width;
    scene.camera.height = height;
    scene.samples = samples;
    Image img(width, height, scene.bg_color);

    if (scene.ray_depth != 0) {  // run_raytracer's early-out, raytracer.h:630
        // Host-side BVH builds stay the reference's code, but only the light BVH is needed: its object order is what
        // bvh_mix_dist::sample indexes (raytracer.h:355-361).  The scene BVH the GPU traverses is the library's own
        // (include/rt_gpu.h: scene_bvh.n_nodes == 0), so the reference's 0.85 s scene build (260k triangles) is skipped
        // unless RT_HOST_SCENE_BVH=1 asks for the reference's tree to be built and passed (RT_KEEP_HOST_BVH=1 makes the
        // library traverse it as is).
        const bool host_tree = env_uint("RT_HOST_SCENE_BVH", 0) != 0;
        std::unique_ptr<RaytracerStaticContext> ctx;
        BVH light_only;
        rt_flatten::FlatScene flat;
        if (host_tree) {
            ctx.reset(new RaytracerStaticContext(scene));
            rt_flatten::flatten(scene, *ctx, flat);
        } else {
            light_only = rt_flatten::build_light_bvh(scene);
            rt_flatten::flatten(scene, nullptr, light_only, flat);
        }
        clock.lap("host BVH + flatten");

        rt_gpu_ctx *gpu = nullptr;
        check(rt_gpu_create(&gpu, static_cast<int>(env_uint("RT_GPUS", 1)), 0), "rt_gpu_create");
        clock.lap("rt_gpu_create (CUDA init)");
        check(rt_gpu_upload_scene(gpu, &flat.desc), "rt_gpu_upload_scene");
        clock.lap("rt_gpu_upload_scene");
        render_into(gpu, width, height, samples, img, &flat.desc.camera);
        clock.lap("render + readback + set_pixel");
        if (aov_samples) {  // RT_PROJECTION was validated by render_into
            const char *projection = std::getenv("RT_PROJECTION");
            rt_projection proj{};
            const bool projected = projection && *projection && parse_projection(projection, proj);
            rt_aov::render_and_write(gpu, width, height, aov_samples, env_uint("RT_SEED", 0), env_uint("RT_PATHS", 128u << 20), &flat.desc.camera,
                                     projected ? &proj : nullptr, argv[5]);
            clock.lap("AOV render + PFMs");
        }
        rt_gpu_destroy(gpu);
        clock.lap("rt_gpu_destroy");
    }

    if (scene.ray_depth == 0 && aov_samples)  // nothing is rendered: the buffers are 0
        rt_aov::render_and_write(nullptr, width, height, aov_samples, 0, 0, nullptr, nullptr, argv[5]);
    write_image(img, argv[5]);
    clock.lap("Image::write");
    return EXIT_SUCCESS;
} catch (std::runtime_error &err) {
    std::cerr << err.what() << std::endl;
    return EXIT_FAILURE;
}
