/*
 * rt_gpu.h — C ABI of the B200 path-tracing backend.
 *
 * This is the drop-in boundary for the per-pixel Monte-Carlo integrator of
 * firelion9/raytracing-course-hw-public.  The reference has no FFI of its own;
 * the seam is the single call `run_raytracer(scene, img)` at
 * src/main.cpp:37 (definition src/raytracer.h:629-674).  A host that keeps the
 * reference's loader (src/scene.h:183), BVH build (src/bvh.h:368) and image
 * writer (src/image.h:34) replaces that one call by
 *
 *     rt_gpu_create -> rt_gpu_upload_scene -> rt_gpu_render -> rt_gpu_readback
 *
 * and then feeds the float means to Image::set_pixel (src/image.h:40), so the
 * tonemap / gamma / PPM path stays the reference's own code.
 *
 * Conventions: plain C, POD structs, caller-owned host pointers that are only
 * read during the call (everything is copied to the device), int return codes
 * (0 = ok, negative = rt_status), no exceptions cross the boundary, one caller
 * thread per handle.  There is no CPU fallback: every entry point fails with
 * RT_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef RT_GPU_H
#define RT_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_GPU_ABI_VERSION 1

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID_ARG = -1,
    RT_ERR_NO_DEVICE = -2,  /* no CUDA device / driver: there is no CPU path */
    RT_ERR_CUDA = -3,       /* a CUDA runtime call failed; see rt_gpu_last_error */
    RT_ERR_NO_SCENE = -4,   /* render/readback before upload */
    RT_ERR_NO_RENDER = -5,  /* readback before render */
    RT_ERR_NCCL = -6,       /* multi-device reduce failed / NCCL not loadable */
    RT_ERR_BAD_SCENE = -7,  /* inconsistent rt_scene_desc (ids out of range ...) */
    RT_ERR_OOM = -8
} rt_status;

#define RT_NO_CHILD 0xFFFFFFFFu /* mirrors NO_CHILD, src/bvh.h:154 */

/* Mirror of `BVHNode` (src/bvh.h:157-163): 40 bytes, same field order, so a
 * reference host can pass `bvh.nodes.data()` without conversion.  A node is
 * either inner (two children, obj_begin == obj_end) or a leaf (no children,
 * objects [obj_begin, obj_end) of the BVH's object order). */
typedef struct rt_bvh_node {
    float bmin[3];
    float bmax[3];
    uint32_t left_child;
    uint32_t right_child;
    uint32_t obj_begin;
    uint32_t obj_end;
} rt_bvh_node;

/* One BVH in the reference's representation (src/bvh.h:165-168).  `objects`
 * replaces the `const Object*` vector by indices into scene.objects order. */
typedef struct rt_bvh_desc {
    uint32_t n_nodes;
    uint32_t root;          /* RT_NO_CHILD when the BVH is empty */
    uint32_t n_objects;
    uint32_t _pad;
    const rt_bvh_node *nodes;
    const uint32_t *objects; /* n_objects ids into the triangle arrays */
} rt_bvh_desc;

/* Mirror of `geometry::material` (src/geometry.h:604-614) with the Texture
 * pointers replaced by indices; -1 selects the built-in 1x1 default
 * (WHITE_TEXTURE, or NORMAL_UP for normal_tex; src/geometry.h:601-602). */
typedef struct rt_material {
    float color[4];
    float emission[3];
    float roughness;
    float metallic;
    float ior;
    int32_t color_tex;
    int32_t emissive_tex;
    int32_t metallic_roughness_tex;
    int32_t normal_tex;
} rt_material;

/* Texture = RGBA8 texels, row-major, `offset` bytes into `texels`.  The
 * reference keeps float4 texels that are exactly u8/255 (src/geometry.h:592-595)
 * so 8-bit storage loses nothing. */
typedef struct rt_texture {
    uint32_t width;
    uint32_t height;
    uint64_t offset;
} rt_texture;

/* Camera (src/scene.h:60-72) without width/height, which are render params. */
typedef struct rt_camera {
    float position[3];
    float right[3];
    float up[3];
    float forward[3];
    float fov_x;
} rt_camera;

/* The flattened scene a host builds from the reference structures
 * (Scene src/scene.h:74-90, RaytracerStaticContext src/raytracer.h:434-455). */
typedef struct rt_scene_desc {
    uint32_t abi_version;     /* RT_GPU_ABI_VERSION */
    uint32_t n_tris;          /* scene.objects.size() */
    rt_camera camera;
    float bg_color[3];        /* Scene::bg_color, constant sky (src/main.cpp:28) */
    /* compile-time knobs of src/config.h, passed as data */
    float eps;                /* EPS = 1e-4, config.h:15 */
    float min_roughness;      /* MIN_ROUGHNESS = 0.04, config.h:20 */
    float vndf_factor;        /* VNDF_factor = 1/3, config.h:26 */
    uint32_t ray_depth;       /* Scene::ray_depth = DEFAULT_RAY_DEPTH = 8 */
    uint32_t n_materials;
    uint32_t n_textures;
    uint32_t flags;           /* RT_SCENE_* bits; 0 = defaults */
    uint32_t env_texture;     /* 0: constant sky = bg_color (HEAD: USE_ENV_MAP = false, src/config.h:36).  k + 1:
                                 textures[k] is the equirectangular environment map `Scene::bg`, looked up by
                                 Scene::bg_at (src/scene.h:83-89) and scaled by bg_color */
    uint64_t texel_bytes;
    /* per-triangle arrays in scene.objects order (Object, geometry.h:639-659) */
    const float *tri_pos;          /* n_tris*9: a,b,c            */
    const float *tri_normals;      /* n_tris*9: per-vertex normals */
    const float *tri_uv;           /* n_tris*6: per-vertex uv    */
    const float *tri_tangents;     /* n_tris*9 or NULL => (1,0,0) */
    const uint32_t *tri_material;  /* n_tris ids into materials  */
    const rt_material *materials;
    const rt_texture *textures;
    const uint8_t *texels;
    rt_bvh_desc scene_bvh;         /* over all triangles (raytracer.h:441-443).  OPTIONAL: n_nodes == 0 (root RT_NO_CHILD,
                                      no arrays) leaves the build to the library, which rebuilds the tree anyway unless
                                      RT_SCENE_KEEP_HOST_BVH is set — a host then skips its own scene-BVH build
                                      (0.85 s for 260k triangles with the reference's builder, bvh.h:262-393) */
    rt_bvh_desc light_bvh;         /* over emission != 0 (raytracer.h:444-447): REQUIRED when the scene has emitters — its
                                      object order is the order bvh_mix_dist::sample indexes (raytracer.h:355-361) */
} rt_scene_desc;

/* rt_scene_desc.flags */
#define RT_SCENE_KEEP_HOST_BVH 1u /* traverse scene_bvh exactly as passed; default: the library rebuilds the
                                     scene BVH over the same triangles with its own SAH builder (closest hits do
                                     not depend on the tree; the reference's builder minimises a mis-stated
                                     surface area, src/geometry.h:419-421, and costs ~25 % more work per ray) */

typedef enum rt_render_mode {
    RT_MODE_BEAUTY = 0,      /* jittered Monte-Carlo estimate (render_pixel, raytracer.h:618) */
    RT_MODE_PRIMARY_IDS = 1  /* pixel-centre rays (gen_ray, raytracer.h:516) -> closest triangle id */
} rt_render_mode;

typedef struct rt_render_params {
    uint32_t width;
    uint32_t height;
    uint32_t samples;        /* total spp of the image */
    uint32_t sample_begin;   /* this call renders samples [sample_begin, sample_end) of every pixel */
    uint32_t sample_end;     /* 0 => samples */
    uint32_t mode;           /* rt_render_mode */
    uint64_t seed;           /* Philox key */
    uint32_t max_paths_in_flight; /* 0 => default: 512 Mi paths (140 B of queue state each = 75 GB), at most half of the
                                     free device memory; callers that share the device (torch, NCCL) pass a bound */
    uint32_t flags;          /* RT_FLAG_* */
    uint32_t pixel_begin;    /* this call renders the row-major pixels [pixel_begin, pixel_end) only (the other */
    uint32_t pixel_end;      /* pixels' sums stay 0 / untouched); 0 => width * height.  Image-tile split. */
} rt_render_params;

#define RT_FLAG_ACCUMULATE 1u /* add to the existing sums instead of clearing them */

/* Work counters of the last render (all devices summed). */
typedef struct rt_stats {
    uint64_t samples;          /* pixel-samples traced */
    uint64_t extension_rays;   /* closest-hit traversals (cast_ray, raytracer.h:540) */
    uint64_t light_pdf_rays;   /* all-hit light-BVH traversals (bvh_mix_dist::pdf, raytracer.h:363) */
    uint64_t shades;           /* shade() evaluations incl. alpha pass-throughs */
    double render_ms;          /* device time of rt_gpu_render (CUDA events), max over devices */
    double reduce_ms;          /* device time of the multi-device reduce (0 for one device) */
    double kernel_ms[8];       /* per-kernel device time: 0 generate 1 extend 2 shade 3 accumulate 4 ids 5 light pdf; filled only with RT_PROFILE_KERNELS */
    uint64_t kernel_launches;  /* kernels launched by the last rt_gpu_render */
} rt_stats;

/* ---- course text scenes (sample_data scene-NNN.txt, homebrew_primitives) ----------------------------------
 * PARITY UNPINNED: the reference at HEAD cannot load or render these (no parser, triangle-only geometry,
 * no delta lights, no refraction; SURVEY.md section 0).  The structures follow the file grammar; the
 * semantics are documented in csrc/text_core.cuh.  Scenes are tiny (<= RT_TEXT_MAX_PRIMS primitives), so
 * the device intersects every primitive per ray (planes are unbounded: no BVH). */
#define RT_TEXT_MAX_PRIMS 256
#define RT_TEXT_MAX_LIGHTS 64
#define RT_TEXT_MAX_DEPTH 16

enum { RT_PRIM_PLANE = 0, RT_PRIM_ELLIPSOID = 1, RT_PRIM_BOX = 2, RT_PRIM_TRIANGLE = 3 };
enum { RT_MAT_DIFFUSE = 0, RT_MAT_METALLIC = 1, RT_MAT_DIELECTRIC = 2 };
enum { RT_LIGHT_DIRECTIONAL = 0, RT_LIGHT_POINT = 1 };
enum { RT_SHADE_FLAT = 0,     /* colour of the nearest primitive (scene-000.txt) */
       RT_SHADE_WHITTED = 1,  /* ambient + delta lights + mirror + Fresnel refraction, RAY_DEPTH (scene-001..004) */
       RT_SHADE_PATH = 2 };   /* Monte-Carlo path tracing, SAMPLES, EMISSION (practice3_*, practice5_*) */

typedef struct rt_text_prim {
    uint32_t kind;      /* RT_PRIM_* */
    uint32_t material;  /* RT_MAT_* */
    float param[9];     /* PLANE: normal; ELLIPSOID: semi-axes; BOX: half extents; TRIANGLE: three vertices */
    float position[3];  /* POSITION (default 0) */
    float rotation[4];  /* ROTATION x y z w (default 0 0 0 1), src/geometry.h:154-156 */
    float color[3];     /* COLOR */
    float emission[3];  /* EMISSION */
    float ior;          /* IOR */
} rt_text_prim;

typedef struct rt_text_light {
    uint32_t kind;         /* RT_LIGHT_* */
    float intensity[3];    /* LIGHT_INTENSITY */
    float vec[3];          /* LIGHT_DIRECTION (towards the light) or LIGHT_POSITION */
    float attenuation[3];  /* LIGHT_ATTENUATION c0 c1 c2: I / (c0 + c1 r + c2 r^2) */
} rt_text_light;

typedef struct rt_text_scene {
    uint32_t abi_version;  /* RT_GPU_ABI_VERSION */
    uint32_t width, height;     /* DIMENSIONS (informative; rt_render_params decides) */
    uint32_t ray_depth;         /* RAY_DEPTH, default 1 (Scene::ray_depth, src/scene.h:76) */
    uint32_t samples;           /* SAMPLES, default 1 (Scene::samples, src/scene.h:77) */
    uint32_t shading;           /* RT_SHADE_* */
    uint32_t n_prims, n_lights;
    float bg_color[3];          /* BG_COLOR */
    float ambient[3];           /* AMBIENT_LIGHT */
    rt_camera camera;
    float eps;                  /* 1e-4, src/config.h:15 */
    const rt_text_prim *prims;
    const rt_text_light *lights;
} rt_text_scene;

typedef struct rt_gpu_ctx rt_gpu_ctx;

/* n_gpus devices starting at first_device (single-process multi-device: one
 * stream per device, ncclReduce to device 0).  A render splits the SAMPLES of
 * every pixel over the devices; when there are fewer samples than devices it
 * splits the IMAGE into contiguous pixel ranges instead (all samples each).  Use n_gpus = 1 and the rank's
 * own device when the caller runs one process per GPU. */
int rt_gpu_create(rt_gpu_ctx **out, int n_gpus, int first_device);
void rt_gpu_destroy(rt_gpu_ctx *ctx);

int rt_gpu_upload_scene(rt_gpu_ctx *ctx, const rt_scene_desc *scene);

/* Upload a course text scene instead of a triangle scene; rt_gpu_render / rt_gpu_readback then work on it
 * (RT_MODE_PRIMARY_IDS gives the primitive index per pixel).  Parity unpinned, see above. */
int rt_gpu_upload_text_scene(rt_gpu_ctx *ctx, const rt_text_scene *scene);

/* Asynchronous with respect to the host only inside the call: returns after
 * the device work (and, for n_gpus > 1, the reduce to device 0) completed. */
int rt_gpu_render(rt_gpu_ctx *ctx, const rt_render_params *params);

/* rgb_mean: width*height*3 floats = per-pixel sum / samples (the argument of
 * Image::set_pixel, image.h:40); prim_ids: width*height int32 (scene.objects
 * index of the primary hit, -1 on miss; only after RT_MODE_PRIMARY_IDS).
 * Either pointer may be NULL. */
int rt_gpu_readback(rt_gpu_ctx *ctx, float *rgb_mean, int32_t *prim_ids, rt_stats *stats);

/* Device pointer of device 0's per-pixel float sums (width*height*4 floats,
 * rgb + w) so that a one-process-per-GPU caller can hand it to its own
 * collective (e.g. torch.distributed.reduce over NCCL) before readback.  w is 0
 * after rt_gpu_render; after rt_gpu_render_adaptive it holds Q = sum of y^2 over
 * the pixel's samples, y = (r + g + b) / 3 of each (NaN-scrubbed) sample, and the
 * rgb sums are over per-pixel sample counts (rt_gpu_readback_adaptive). */
int rt_gpu_accum_device_ptr(rt_gpu_ctx *ctx, void **dptr, size_t *n_floats);

/* Device-side tonemap + quantise of the current sums (image.h:49-82):
 * rgb8 = width*height*3 bytes, ready to follow the "P6" header. */
int rt_gpu_readback_rgb8(rt_gpu_ctx *ctx, uint8_t *rgb8);

/* ---- adaptive sampling -------------------------------------------------------------------------------------
 * rt_gpu_render_adaptive traces every pixel of [pixel_begin, pixel_end) until its noise reaches a target:
 * params->samples is the MAXIMUM spp.  Round 0 gives every pixel min_samples samples; every later round gives
 * step_samples more to each pixel that has not converged (the last round clipped at samples).  A pixel always has
 * the sample prefix [0, n_p), so the image is, pixel by pixel, a fixed render truncated at that pixel's count.
 * After n samples with S = sum y, Q = sum y^2 (y = (r + g + b) / 3 of each sample), in double precision:
 *     m = S / n,  var = max(Q / n - m^2, 0) * n / (n - 1),  err = sqrt(var / n) / (m + abs_floor)
 * and the pixel stops once err <= rel_error (rel_error = 0: never early; with min_samples == samples that is a
 * fixed render that also yields the error map).  Afterwards rt_gpu_readback returns sum / n_p per pixel (0 where
 * n_p = 0, i.e. outside the range), rt_gpu_readback_rgb8 tonemaps the same means and stats.samples = sum of n_p.
 * RT_ERR_INVALID_ARG for sample_begin / sample_end != 0, RT_FLAG_ACCUMULATE, RT_MODE_PRIMARY_IDS, samples < 2,
 * min_samples < 2, step_samples == 0, abs_floor <= 0, a text scene, or a (per-device) pixel range larger than one
 * batch of max_paths_in_flight paths.  A multi-device handle splits the range into contiguous parts, one per
 * device; the image equals the one-device image bit for bit.  RT_FLAG_ACCUMULATE on a render that follows an
 * adaptive one fails with RT_ERR_INVALID_ARG (the sums have per-pixel counts); without it a render behaves as on a
 * fresh handle. */
typedef struct rt_adaptive_params {
    uint32_t min_samples;   /* first round, every pixel of the range; >= 2 */
    uint32_t step_samples;  /* added per later round to every pixel not yet converged; >= 1 */
    float rel_error;        /* stop a pixel once err <= rel_error (0: never stop early) */
    float abs_floor;        /* > 0: keeps near-black pixels from chasing relative noise */
} rt_adaptive_params;

int rt_gpu_render_adaptive(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_adaptive_params *ap);

/* After rt_gpu_render_adaptive: per-pixel sample counts (width*height uint32) and the err each pixel last had
 * (width*height float; 0 outside the range); either may be NULL.  After rt_gpu_render_views_adaptive: the same for
 * the stacked image (n_views*width*height each).  RT_ERR_NO_RENDER after any other render. */
int rt_gpu_readback_adaptive(rt_gpu_ctx *ctx, uint32_t *sample_counts, float *rel_error);

/* ---- multi-view rendering ----------------------------------------------------------------------------------
 * rt_gpu_render_views traces n_views cameras over the uploaded triangle scene in one render.  The views of
 * width x height are stacked into one image of width x (n_views * height): pixel v * width * height + y * width + x
 * is pixel (x, y) of view v.  Afterwards rt_gpu_readback returns n_views * width * height * 3 floats (view-major)
 * and, after RT_MODE_PRIMARY_IDS, n_views * width * height ids; rt_gpu_readback_rgb8 returns
 * n_views * width * height * 3 bytes; rt_gpu_accum_device_ptr reports n_views * width * height * 4 floats;
 * stats.samples counts every view.  rt_render_params keep their meaning; pixel_begin / pixel_end index the stacked
 * image [0, n_views * width * height), and a multi-device handle splits it like any image.
 * Pixel p of view v is keyed (Philox) as pixel (view_base + v) * width * height + p, so:
 *   - one view with the scene's own camera and view_base = 0 is rt_gpu_render, bit for bit;
 *   - view v of a call is a one-view call with view_base = v (bit for bit when both run in the same batches),
 * and how a camera path is split into calls does not change a frame.
 * RT_ERR_INVALID_ARG for n_views == 0, cameras == NULL, a non-finite camera value, (view_base + n_views) * width *
 * height > 2^32, a stacked image of more than 2^31 - 1 pixels, a text scene, and RT_FLAG_ACCUMULATE unless the
 * previous render had the same width, height and n_views (rt_gpu_render counts as one view; this holds in both
 * directions).  Without the flag, a render behaves as on a fresh handle.  Adaptive sampling over views is not
 * offered by this call: rt_gpu_readback_adaptive returns RT_ERR_NO_RENDER after it (rt_gpu_render_views_adaptive
 * below is the adaptive form). */
typedef struct rt_views {
    uint32_t n_views;          /* >= 1 */
    uint32_t view_base;        /* Philox pixel key of pixel p of view v = (view_base + v) * width * height + p */
    const rt_camera *cameras;  /* n_views cameras; same convention as rt_scene_desc.camera (fov_y from width / height) */
} rt_views;

int rt_gpu_render_views(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views);

/* Adaptive multi-view rendering: rt_gpu_render_adaptive over the stacked image of rt_gpu_render_views.  The image,
 * pixel range and keys are rt_gpu_render_views' (pixel_begin / pixel_end index [0, n_views * width * height); pixel p
 * of view v is keyed (view_base + v) * width * height + p); the rounds, the rule, params->samples as the maximum spp
 * and the sample prefix [0, n_p) of every pixel are rt_gpu_render_adaptive's.  So:
 *   - one view with the scene's own camera and view_base = 0 is rt_gpu_render_adaptive, bit for bit;
 *   - view v of a call is a one-view call with view_base = v (bit for bit when both run in the same batches);
 *   - a pixel with count n equals rt_gpu_render_views of samples [0, n) summed in the same sample ranges.
 * Afterwards rt_gpu_readback returns n_views * width * height * 3 means (sum / n_p, view-major), rt_gpu_readback_rgb8
 * n_views * width * height * 3 bytes, rt_gpu_readback_adaptive n_views * width * height counts and errors,
 * rt_gpu_accum_device_ptr reports n_views * width * height * 4 floats, and stats.samples = sum of n_p.
 * RT_ERR_INVALID_ARG for everything either call refuses: a null argument, a text scene, n_views == 0, cameras == NULL,
 * a non-finite camera value, (view_base + n_views) * width * height > 2^32, a stacked image of more than 2^31 - 1
 * pixels, RT_MODE_PRIMARY_IDS, samples < 2, sample_begin / sample_end != 0, RT_FLAG_ACCUMULATE, bad
 * rt_adaptive_params, an illegal pixel range, or a (per-device) range larger than one batch of max_paths_in_flight
 * paths.  A multi-device handle splits the stacked range into contiguous parts, as rt_gpu_render_adaptive does.  The
 * sums have per-pixel counts afterwards: RT_FLAG_ACCUMULATE on the next rt_gpu_render / rt_gpu_render_views fails with
 * RT_ERR_INVALID_ARG; without it a render behaves as on a fresh handle.  A round of k samples runs in ceil(k / k_max)
 * batches, k_max = paths per batch / pixels of the (per-device) range: more views mean more batches per round. */
int rt_gpu_render_views_adaptive(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views,
                                 const rt_adaptive_params *ap);

/* ---- camera projections -----------------------------------------------------------------------------------------
 * rt_gpu_render_projected renders the views of rt_views, each through its own projection of its camera (position and
 * right / up / forward basis; fov_x is used by the pinhole and thin-lens kinds only).  For image point (px, py) in
 * pixels (centres at + 0.5), with W x H the size of one view:
 *   RT_PROJ_PINHOLE        the camera ray of rt_gpu_render_views, bit for bit;
 *   RT_PROJ_THIN_LENS      d = the pinhole direction; focus = position + d * focus_distance / dot(d, forward) (the plane
 *                          in focus lies focus_distance along forward); the ray starts at a uniform point of the lens disc
 *                          of aperture_radius spanned by right and up and passes through focus.  aperture_radius == 0 is
 *                          the pinhole, bit for bit;
 *   RT_PROJ_ORTHOGRAPHIC   origin position + a * right - b * up with a = (2 px / W - 1) * half_width,
 *                          b = (2 py / H - 1) * half_height (glTF xmag / ymag), direction forward (normalised);
 *   RT_PROJ_EQUIRECT       u = (px - 0.5) / W, v = (py - 0.5) / H, phi = (u - 0.5) * 2 pi, theta = (0.5 - v) * pi,
 *                          d = cos(theta) sin(phi) * right + sin(theta) * up + cos(theta) cos(phi) * forward, normalised:
 *                          the full sphere, forward at the image centre.  With forward = +x, right = +z, up = +y a view
 *                          of the environment map's size looks up texel (i, j) at the centre of pixel (i, j).
 * Lens samples use their own Philox stream (counter word 2 = 0xFFFFFFFE); every other random number of a path is the
 * one rt_gpu_render_views draws.  RT_MODE_PRIMARY_IDS traces pixel centres through the lens centre.
 * ap == NULL: the contract of rt_gpu_render_views (image, keys, readbacks, accumulation, multi-device split).
 * ap != NULL: the contract of rt_gpu_render_views_adaptive.  So all-pinhole projections give exactly those calls.
 * RT_ERR_INVALID_ARG for everything the corresponding view call refuses, and for projections == NULL, an unknown kind,
 * a non-finite field, aperture_radius < 0, focus_distance <= 0 with aperture_radius > 0, and half_width or
 * half_height <= 0 for RT_PROJ_ORTHOGRAPHIC.  Fields a kind does not use are ignored. */
#define RT_PROJ_PINHOLE 0u
#define RT_PROJ_THIN_LENS 1u
#define RT_PROJ_ORTHOGRAPHIC 2u
#define RT_PROJ_EQUIRECT 3u

typedef struct rt_projection {
    uint32_t kind;          /* RT_PROJ_* */
    float aperture_radius;  /* thin lens: radius of the lens disc (world units); 0 = pinhole */
    float focus_distance;   /* thin lens: distance of the plane in focus along forward; > 0 when aperture_radius > 0 */
    float half_width;       /* orthographic: half the view's extent along right (glTF xmag); > 0 */
    float half_height;      /* orthographic: half the view's extent along up (glTF ymag); > 0 */
} rt_projection;

int rt_gpu_render_projected(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views,
                            const rt_projection *projections /* n_views */, const rt_adaptive_params *ap /* NULL = fixed */);

/* ---- animated geometry ------------------------------------------------------------------------------------------
 * rt_gpu_update_geometry moves the triangles of the uploaded scene in place: positions, normals, tangents and the light
 * BVH are replaced, with the meaning they have in rt_scene_desc; triangles, uv, materials, textures, camera, sky, flags
 * and ray depth stay as uploaded.  The scene BVH keeps its topology (binary tree, triangle order, and which binary nodes
 * form each 4-wide node with which children): every box is refit to the new positions and re-quantised.  So:
 *   - the link words of rt_gpu_debug_get_bvh selector 3 and the counts of selector 0 do not change, nor does the
 *     traversal-stack need (an update never fails on RT_EXT_STACK_CAP);
 *   - upload(A); update(B); update(A) leaves the device scene byte-identical to upload(A), and update(A) right after
 *     upload(A) changes nothing;
 *   - afterwards selectors 1..4 describe the refit tree: binary boxes are the exact union of what lies below them,
 *     quantised boxes contain every vertex below them and the device triangles hold the new positions.
 * A tree refit far from the positions it was built for traces slower (its boxes overlap more); a re-upload builds a
 * new tree.  The light side becomes what rt_gpu_upload_scene makes of light_bvh and the new positions: light nodes,
 * light triangles, the sampling list, the light normals and areas, and the light box.
 * The last render's sums, counts, ids and stats are left alone, and so are the accumulation rules: RT_FLAG_ACCUMULATE
 * on the next render adds samples of the new geometry to the old sums (motion blur by sub-frame accumulation).
 * RT_ERR_NO_SCENE before any upload.  RT_ERR_INVALID_ARG, with the scene untouched, for a null argument, a text scene,
 * n_tris != the uploaded n_tris, a null tri_pos or tri_normals with n_tris > 0, a light BVH with another n_objects or
 * with ids or links out of range, and a scene whose tree was not built on the device (uploaded with
 * RT_SCENE_KEEP_HOST_BVH, RT_KEEP_HOST_BVH or RT_HOST_BUILD set, or by the 8-wide library: those trees live on the
 * host; re-upload instead).  RT_ERR_BAD_SCENE for a non-finite vertex or a node that cannot be quantised: these are
 * found on the device after the arrays were overwritten, so the handle then holds no scene and renders return
 * RT_ERR_NO_SCENE until the next upload.  Every device of a handle is updated; the call returns after the device
 * work is complete. */
typedef struct rt_geometry_update {
    uint32_t n_tris;            /* must equal the uploaded scene's n_tris */
    uint32_t _pad;
    const float *tri_pos;       /* n_tris*9, scene.objects order; required when n_tris > 0 */
    const float *tri_normals;   /* n_tris*9; required when n_tris > 0 */
    const float *tri_tangents;  /* n_tris*9 or NULL => (1,0,0), as in rt_scene_desc */
    rt_bvh_desc light_bvh;      /* the light BVH over the NEW positions (what rt_scene_desc.light_bvh would be); same
                                   n_objects as uploaded; empty when the scene has no emitters */
} rt_geometry_update;

int rt_gpu_update_geometry(rt_gpu_ctx *ctx, const rt_geometry_update *u);

/* Diagnostic (tests): the scene BVH the library built on the device during the last rt_gpu_upload_scene (with the
 * boxes of any rt_gpu_update_geometry since).
 * which = 0: uint32[8] {n_tris, binary node slots, 4-wide nodes, root link, worst-case traversal stack need, depth of
 * the binary tree, 1 if built on the device, levels of the top-down phase}; 1: rt_bvh_node[slots] (the binary tree in the
 * slot layout left = i + 1, right = i + 2 * n_left; unused slots are undefined); 2: uint32[n_tris] scene.objects id at
 * each BVH position; 3: the 4-wide quantised nodes (64 B each); 4: the device triangles (64 B each, n_tris + 1).
 * dst == NULL only reports the size in *bytes.  Selectors 1..4 are empty when the host built the tree. */
int rt_gpu_debug_get_bvh(rt_gpu_ctx *ctx, int which, void *dst, size_t *bytes);

/* Diagnostic (tests): the light pdf (bvh_mix_dist::pdf, the 1 / n_lights factor included) of n caller rays, as the next
 * k_shade reads it from the queue for a pending ray: rays is n x 6 floats (origin, then direction as the renderer stores
 * it), pdf receives n floats.  The default library appends the rays to a pending queue with k_shade's own append (box of
 * all lights: 0 on a miss, else listed) and runs k_lightpdf_list; the 8-wide library runs k_extend8 over them as a
 * bounce > 0.  Device 0 only; buffers are allocated per call and freed before it returns, which is after the device work.
 * RT_ERR_NO_SCENE before any upload; RT_ERR_INVALID_ARG for a null pointer (rays / pdf with n > 0) or a text scene.  A
 * scene without emitters gives zeros and launches nothing. */
int rt_gpu_debug_light_pdf(rt_gpu_ctx *ctx, uint64_t n, const float *rays, float *pdf);

/* Per-kernel timing (serialises launches with events; off by default). */
int rt_gpu_set_profiling(rt_gpu_ctx *ctx, int enable);

/* Diagnostic: measured FP32 FMA rate of device 0 in TFLOP/s (dependent-chain-free FFMA loop on every
 * SM) — the denominator of the FP32 roofline the traversal / shading kernels are reported against. */
int rt_gpu_fp32_peak(rt_gpu_ctx *ctx, double *tflops);

const char *rt_gpu_last_error(void);
int rt_gpu_device_count(void);
int rt_gpu_abi_version(void);

#ifdef __cplusplus
}
#endif

#endif /* RT_GPU_H */
