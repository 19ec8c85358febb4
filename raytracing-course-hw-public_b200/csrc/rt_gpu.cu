// rt_gpu.cu — implementation of the C ABI in include/rt_gpu.h on top of the wavefront kernels.
//
// One DeviceState per GPU (own stream, own copy of the scene, own queues).  A render splits the
// sample range across the devices of the handle (sample-split; SURVEY.md 8(e); image tiles when there
// are fewer samples than devices), every device runs its batches asynchronously on its stream, and
// for more than one device the per-pixel float sums are merged with a single ncclReduce(sum) to
// device 0.  rt_gpu_upload_scene re-packs on the host (own SAH tree, 4-wide collapse, quantisation).  NCCL is resolved with dlopen at the first
// multi-device create so that single-device users never need the library.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "extend8.cuh"
#ifndef RT_EXT_WIDE8
#define RT_EXT_WIDE8 0  // 1: k_extend8 over 8-wide nodes (extend8.cuh) instead of k_extend over 4-wide ones
#endif
#if RT_EXT_WIDE8
#define RT_K_EXTEND rt::k_extend8
#else
#define RT_K_EXTEND rt::k_extend
#endif
#include "text_kernels.cuh"
#include "repack.h"
#include "gpu_build.cuh"
#include "adaptive.cuh"
#include "views.cuh"
#include "projection.cuh"
#include "aov.cuh"
#include "rt_gpu.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}

#define CU_CHECK(expr)                                                                                       \
    do {                                                                                                     \
        cudaError_t _e = (expr);                                                                             \
        if (_e != cudaSuccess)                                                                               \
            return fail(_e == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA,                          \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                 \
    } while (0)

// ---- minimal NCCL binding (dlopen) ---------------------------------------------------------------
typedef struct ncclComm *ncclComm_t;
struct NcclApi {
    void *handle = nullptr;
    int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*Reduce)(const void *, void *, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (handle) return true;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) return false;
        CommInitAll = reinterpret_cast<decltype(CommInitAll)>(dlsym(handle, "ncclCommInitAll"));
        CommDestroy = reinterpret_cast<decltype(CommDestroy)>(dlsym(handle, "ncclCommDestroy"));
        Reduce = reinterpret_cast<decltype(Reduce)>(dlsym(handle, "ncclReduce"));
        GroupStart = reinterpret_cast<decltype(GroupStart)>(dlsym(handle, "ncclGroupStart"));
        GroupEnd = reinterpret_cast<decltype(GroupEnd)>(dlsym(handle, "ncclGroupEnd"));
        GetErrorString = reinterpret_cast<decltype(GetErrorString)>(dlsym(handle, "ncclGetErrorString"));
        return CommInitAll && CommDestroy && Reduce && GroupStart && GroupEnd;
    }
};
NcclApi g_nccl;
constexpr int kNcclUint32 = 3;   // ncclUint32
constexpr int kNcclFloat32 = 7;  // ncclFloat32
constexpr int kNcclSum = 0;      // ncclSum

template <class T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    int alloc(size_t count) {
        if (count <= n && p) return RT_OK;
        release();
        if (count == 0) return RT_OK;
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&p), count * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr;
            return fail(RT_ERR_OOM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
        }
        n = count;
        return RT_OK;
    }
    int upload(const std::vector<T> &v, cudaStream_t s) {
        if (int rc = alloc(std::max<size_t>(v.size(), 1))) return rc;
        if (!v.empty()) CU_CHECK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
        return RT_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

constexpr size_t kBytesPerPath = 8 * sizeof(float4) + 3 * sizeof(float);  // q_o, q_d, q_thr (x2 parities) + hit + rad + lpdf (x2) + light list
constexpr size_t kAovBytesPerPath = 3 * sizeof(float4);                       // an AOV render's slots (aov.cuh), beyond the queues

enum KernelKind { K_GENERATE = 0, K_EXTEND = 1, K_SHADE = 2, K_ACCUMULATE = 3, K_IDS = 4, K_LIGHTPDF = 5, K_COUNT = 8 };

struct DeviceState {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of the triangle attributes while the BVH build runs on `stream`
    cudaStream_t stream2 = nullptr;      // second half of every queue (enqueue_render): its kernels fill the SMs that the
                                         // first half's draining persistent kernel leaves idle, and vice versa
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_light = nullptr;  // cross-stream ordering of the two halves
    cudaEvent_t ev_copied = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_red0 = nullptr, ev_red1 = nullptr;
    // scene
    DevBuf<QNode4> qnodes4, lqnodes4;  // scene BVH and light BVH, 4-wide quantised (both traversed by k_extend)
    DevBuf<QNode8> qnodes8, lqnodes8;  // 8-wide (RT_EXT_WIDE8 builds)
    DevBuf<uint4> q4split;             // both 4-wide node arrays once more, as two halves of 32-byte stride (DBvh::q4lo)
    DevBuf<DTri> tris, ltris, lsample;
    DevBuf<DAttr> attrs;
    DevBuf<DTangent> tangents;
    DevBuf<DLight> light_extra;
    DevBuf<DMat> materials;
    DevBuf<DTex> textures;
    DevBuf<uint32_t> texels;
    DevBuf<float> lut;
    DScene scene;
    // device-side scene build (gpu_build.cuh): H2D copies of the host's arrays, scratch, last result
    DevBuf<float> in_pos, in_nrm, in_uv, in_tan;
    DevBuf<uint32_t> in_mat;
    DevBuf<uint8_t> build_scratch;
    rtb::Counters *h_counters = nullptr;  // pinned
    rtb::Arrays built{};                  // device pointers of the last device build (diagnostics)
    uint32_t built_info[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // n_tris, n_slots, n_wide, root4, stack_need, max_depth, 1 = device build, levels
    int built_parity = 0;
    // refit of that tree (rt_gpu_update_geometry): recorded at the first update after an upload
    DevBuf<uint8_t> refit_scratch;
    rtb::Refit refit{};
    bool refit_ready = false;
    std::vector<uint32_t> refit_lstart, refit_lcount;  // the binary levels of refit.order
    // course text scene (rt_gpu_upload_text_scene)
    DevBuf<rt_text_prim> tprims;
    DevBuf<rt_text_light> tlights;
    DevBuf<uint32_t> temit;
    rtt::TextScene tscene;
    rt_camera tcamera;
    // render state
    // Path-state queues: ONE allocation, carved at fixed 2 MB-aligned offsets (round 1 used nine cudaMallocs of
    // multi-GB arrays, whose relative placement differed from process to process).
    DevBuf<uint8_t> arena;
    size_t queue_cap = 0;  // paths the arena holds
    float4 *qo[2] = {nullptr, nullptr}, *qd[2] = {nullptr, nullptr}, *qthr[2] = {nullptr, nullptr}, *hit = nullptr, *rad = nullptr;
    float *lpdf[2] = {nullptr, nullptr};  // by queue parity, like qo / qd / qthr
    uint32_t *light_list = nullptr;  // RT_LIGHT_KERNEL == 2: queue indices of the pending rays that pass the light box
    DevBuf<float4> accum;
    DevBuf<float> means;   // packed rgb means (rt_gpu_readback)
    DevBuf<uint32_t> counters;
    unsigned long long *h_stats = nullptr;  // pinned: the work counters arrive with the render's own stream sync
    float *h_means = nullptr;               // pinned staging of the readback
    size_t h_means_n = 0;
    void *h_stage = nullptr;                // pinned staging of the scene upload
    size_t h_stage_n = 0;
    int alloc_queues(size_t cap) {
        if (cap <= queue_cap && arena.p) return RT_OK;
        const size_t align = size_t(2) << 20;
        auto up = [&](size_t b) { return (b + align - 1) / align * align; };
        const size_t b16 = up(cap * sizeof(float4)), b4 = up(cap * sizeof(float));
        arena.release();
        queue_cap = 0;
        if (int rc = arena.alloc(8 * b16 + 3 * b4)) return rc;
        uint8_t *p = arena.p;
        if (std::getenv("RT_TIMING"))
            std::fprintf(stderr, "rt_gpu: queue arena %p, %.1f MiB, base mod 512 MiB = %zu MiB\n", static_cast<void *>(p),
                         (8 * b16 + 3 * b4) / 1048576.0, (reinterpret_cast<size_t>(p) >> 20) & 511);
        auto take = [&](size_t b) { uint8_t *r = p; p += b; return r; };
        for (int i = 0; i < 2; ++i) {
            qo[i] = reinterpret_cast<float4 *>(take(b16));
            qd[i] = reinterpret_cast<float4 *>(take(b16));
            qthr[i] = reinterpret_cast<float4 *>(take(b16));
        }
        hit = reinterpret_cast<float4 *>(take(b16));
        rad = reinterpret_cast<float4 *>(take(b16));
        lpdf[0] = reinterpret_cast<float *>(take(b4));
        lpdf[1] = reinterpret_cast<float *>(take(b4));
        light_list = reinterpret_cast<uint32_t *>(take(b4));
        queue_cap = cap;
        return RT_OK;
    }
    DevBuf<unsigned long long> stats;
    // adaptive sampling (rt_gpu_render_adaptive, adaptive.cuh): two active lists (ping-pong), the flag words and their
    // scan, per-pixel sample counts and errors (whole image, 0 outside this device's range), the active count of each
    // list; each round's count travels behind ev_round[round & 1] into the pinned h_active[round & 1]
    DevBuf<uint32_t> alist, awords, acounts, actr;
    DevBuf<float> aerr;
    uint32_t *h_active = nullptr;
    cudaEvent_t ev_round[2] = {nullptr, nullptr};
    size_t apix0 = 0, apix1 = 0;  // the pixel range this device adapted in the last adaptive render
    DevBuf<int32_t> prim_ids;
    DevBuf<uint8_t> rgb8;
    DevBuf<rt::Camera> cams;  // the cameras of the last multi-view render (rt_gpu_render_views), one per view
    DevBuf<rt::Projection> projs;  // their projections when it was rt_gpu_render_projected
    // AOV render (rt_gpu_render_aov, aov.cuh): three float4 slots per path of a batch (aov_cap paths), three float4
    // sums per pixel of the last AOV render, and the means of its readback
    DevBuf<float4> aov_slots, aov_sums;
    size_t aov_cap = 0;
    DevBuf<float> aov_means;
    int extend_blocks = 0, shade_blocks = 0, light_blocks = 0;
    rt::LightBox light_box{};  // box of all light triangles (k_shade tests the rays it queues against it)
    // profiling
    std::vector<std::pair<cudaEvent_t, int>> marks;  // event recorded AFTER a kernel of that kind
    std::vector<cudaEvent_t> event_pool;
    size_t events_used = 0;

    cudaEvent_t next_event() {
        if (events_used == event_pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            event_pool.push_back(e);
        }
        return event_pool[events_used++];
    }
};

}  // namespace

struct rt_gpu_ctx {
    std::vector<std::unique_ptr<DeviceState>> devs;
    std::vector<ncclComm_t> comms;
    bool have_scene = false, have_render = false, profiling = false;
    bool text_scene = false;  // the uploaded scene is a course text scene
    bool adaptive = false;       // the last render was rt_gpu_render_adaptive (rt_gpu_readback_adaptive has data)
    bool adaptive_sums = false;  // the sums are an adaptive render's: per-pixel sample counts, Q in w
    rt_adaptive_params last_adaptive{};
    rt_render_params last{};
    uint32_t last_views = 0;  // views of the last render: 0 = not rt_gpu_render_views (one image, the scene's camera)
    rt_stats stats{};
    uint32_t ray_depth = 0;
    rt::PackedScene packed;  // staging of the last upload, kept so that the next one re-uses its (already touched) memory
    // the last AOV render (rt_gpu_render_aov): its resolved parameters, views (0 = the scene camera), the sample count
    // its readback divides by, and its own stats; rt_gpu_readback_aov returns RT_ERR_NO_RENDER before the first
    bool have_aov = false;
    rt_render_params aov_last{};
    uint32_t aov_views = 0, aov_samples = 0;
    rt_stats aov_stats{};
};

namespace {

// Scene BVH, triangles and attributes built on the device from the host's arrays (gpu_build.cuh).  Fills d.qnodes4,
// d.tris, d.attrs (, d.tangents) and the root link / counts in `info`.
int device_build_scene(DeviceState &d, const rt_scene_desc &sc, double *t_h2d_ms) {
    using namespace rtb;
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t n = sc.n_tris;
    const auto t0 = std::chrono::steady_clock::now();
    // The build needs the positions only; normals, uv, materials and tangents (3/4 of the bytes) are copied on a second
    // stream while it runs and are waited for before they are first read (from pinned host memory the copies are real
    // DMA and overlap; from pageable memory cudaMemcpyAsync stages synchronously and nothing is lost).
    auto h2d = [&](auto &buf, const auto *src, size_t count, cudaStream_t on) -> int {
        if (int rc = buf.alloc(std::max<size_t>(count, 1))) return rc;
        if (count) CU_CHECK(cudaMemcpyAsync(buf.p, src, count * sizeof(*src), cudaMemcpyHostToDevice, on));
        return RT_OK;
    };
    if (int rc = h2d(d.in_pos, sc.tri_pos, static_cast<size_t>(n) * 9, d.stream)) return rc;
    // (the previous render's kernels on d.stream may still read nothing of these buffers: rt_gpu_render is synchronous)
    if (int rc = h2d(d.in_nrm, sc.tri_normals, static_cast<size_t>(n) * 9, d.copy_stream)) return rc;
    if (int rc = h2d(d.in_uv, sc.tri_uv, static_cast<size_t>(n) * 6, d.copy_stream)) return rc;
    if (int rc = h2d(d.in_mat, sc.tri_material, static_cast<size_t>(n), d.copy_stream)) return rc;
    if (sc.tri_tangents)
        if (int rc = h2d(d.in_tan, sc.tri_tangents, static_cast<size_t>(n) * 9, d.copy_stream)) return rc;
    CU_CHECK(cudaEventRecord(d.ev_copied, d.copy_stream));
    if (t_h2d_ms) *t_h2d_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();

    // scratch carved from one allocation
    const size_t n_slots = n ? 2 * static_cast<size_t>(n) - 1 : 0;
    const size_t n_pool = n / kSmall + 2;
    const size_t n_words = (std::max<size_t>(n_slots, n) + 31) / 32 + 8;
    size_t off = 0;
    auto carve = [&](size_t bytes) {
        const size_t at = off;
        off += (bytes + 255) / 256 * 256;
        return at;
    };
    const size_t o_plo = carve(n * sizeof(float4)), o_phi = carve(n * sizeof(float4));
    const size_t o_idx0 = carve(n * 4), o_idx1 = carve(n * 4), o_nof0 = carve(n * 4), o_nof1 = carve(n * 4);
    const size_t o_nodes = carve(std::max<size_t>(n_slots, 1) * sizeof(rt_bvh_node)), o_aux = carve(std::max<size_t>(n_slots, 1) * sizeof(NodeAux));
    const size_t o_bins0 = carve(n_pool * sizeof(BinSlot)), o_bins1 = carve(n_pool * sizeof(BinSlot));
    const size_t o_act0 = carve(n_pool * 4), o_act1 = carve(n_pool * 4), o_small = carve((static_cast<size_t>(n) + 1) * 4);
    const size_t o_words = carve(n_words * 4), o_wscan = carve(n_words * 4);
    const size_t o_last = carve(static_cast<size_t>(n) + 1), o_mark = carve(n_slots + 1), o_need = carve((n_slots + 1) * 4);
    const size_t o_fr0 = carve((static_cast<size_t>(n) + 1) * 4), o_fr1 = carve((static_cast<size_t>(n) + 1) * 4), o_fr2 = carve((static_cast<size_t>(n) + 1) * 4);
    const size_t o_cnt = carve(sizeof(Counters));
    if (int rc = d.build_scratch.alloc(off)) return rc;
    uint8_t *base = d.build_scratch.p;
    if (int rc = d.qnodes4.alloc(std::max<size_t>(n, 1))) return rc;  // a tree over n triangles has fewer than n wide nodes
    if (int rc = d.tris.alloc(static_cast<size_t>(n) + 1)) return rc;
    if (int rc = d.attrs.alloc(std::max<size_t>(n, 1))) return rc;

    Arrays A{};
    A.tri_pos = d.in_pos.p;
    A.tri_normals = d.in_nrm.p;
    A.tri_uv = d.in_uv.p;
    A.tri_tangents = sc.tri_tangents ? d.in_tan.p : nullptr;
    A.tri_material = d.in_mat.p;
    A.n = n;
    A.plo = reinterpret_cast<float4 *>(base + o_plo);
    A.phi = reinterpret_cast<float4 *>(base + o_phi);
    A.idx[0] = reinterpret_cast<uint32_t *>(base + o_idx0);
    A.idx[1] = reinterpret_cast<uint32_t *>(base + o_idx1);
    A.node_of[0] = reinterpret_cast<uint32_t *>(base + o_nof0);
    A.node_of[1] = reinterpret_cast<uint32_t *>(base + o_nof1);
    A.nodes = reinterpret_cast<rt_bvh_node *>(base + o_nodes);
    A.aux = reinterpret_cast<NodeAux *>(base + o_aux);
    A.bins[0] = reinterpret_cast<BinSlot *>(base + o_bins0);
    A.bins[1] = reinterpret_cast<BinSlot *>(base + o_bins1);
    A.active[0] = reinterpret_cast<uint32_t *>(base + o_act0);
    A.active[1] = reinterpret_cast<uint32_t *>(base + o_act1);
    A.small = reinterpret_cast<uint32_t *>(base + o_small);
    A.words = reinterpret_cast<uint32_t *>(base + o_words);
    A.wscan = reinterpret_cast<uint32_t *>(base + o_wscan);
    A.last = base + o_last;
    A.mark = base + o_mark;
    A.need = reinterpret_cast<uint32_t *>(base + o_need);
    A.frontier[0] = reinterpret_cast<uint32_t *>(base + o_fr0);
    A.frontier[1] = reinterpret_cast<uint32_t *>(base + o_fr1);
    A.frontier[2] = reinterpret_cast<uint32_t *>(base + o_fr2);
    A.c = reinterpret_cast<Counters *>(base + o_cnt);
    A.qnodes4 = d.qnodes4.p;
    A.tris = d.tris.p;
    A.attrs = d.attrs.p;
    A.tangents = nullptr;
    cudaStream_t st = d.stream;
    Counters &hc = *d.h_counters;
    auto fetch_counters = [&]() -> int {
        CU_CHECK(cudaMemcpyAsync(&hc, A.c, sizeof(Counters), cudaMemcpyDeviceToHost, st));
        CU_CHECK(cudaStreamSynchronize(st));
        return RT_OK;
    };
    const bool timing = std::getenv("RT_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    std::string phases;
    auto lap = [&](const char *name) {  // RT_TIMING only: serialises the build at the phase boundaries
        if (!timing) return;
        cudaStreamSynchronize(st);
        const auto now = std::chrono::steady_clock::now();
        char buf[64];
        std::snprintf(buf, sizeof buf, " %s %.2f", name, std::chrono::duration<double, std::milli>(now - t_last).count());
        phases += buf;
        t_last = now;
    };
    lap("h2d+alloc");
    d.refit_ready = false;
    std::memset(d.built_info, 0, sizeof d.built_info);
    d.built = A;
    d.built_parity = 0;
    d.built_info[0] = n;
    d.built_info[3] = static_cast<uint32_t>(RT_LINK_NONE);
    d.built_info[6] = 1;
    kb_init<<<1, 1, 0, st>>>(A);
    if (n == 0) {  // empty scene: only the null triangle
        kb_tris<<<1, 256, 0, st>>>(A, 0, 0);
        CU_CHECK(cudaGetLastError());
        CU_CHECK(cudaStreamSynchronize(st));
        return RT_OK;
    }
    const uint32_t g_n = (n + 255) / 256;
    CU_CHECK(cudaMemsetAsync(A.mark, 0, n_slots + 1, st));
    kb_setup<<<g_n, 256, 0, st>>>(A);
    kb_root<<<1, 32, 0, st>>>(A);
    lap("setup");
    // big phase.  The host does not know when the last big node is gone: it asks every other level, starting where a
    // balanced tree over n triangles would first run out of nodes with more than kSmall triangles.
    int first_check = 0;
    while ((static_cast<uint64_t>(kSmall) << (first_check + 1)) < n) ++first_check;
    const uint32_t n_bin_words = (n + 31) / 32;
    const uint32_t g_split = static_cast<uint32_t>((n_pool + 3) / 4);  // one warp per node
    int parity = 0;
    uint32_t level = 0;
    bool attrs_joined = false;
    for (;; ++level) {
        if (level >= RT_STACK_SIZE) return fail(RT_ERR_CUDA, "device BVH build did not terminate");
        if (static_cast<int>(level) >= first_check && ((level - first_check) & 1u) == 0) {
            if (!attrs_joined) {  // the attribute copies have had the top levels' time; the tangent flag rides on this fetch
                CU_CHECK(cudaStreamWaitEvent(st, d.ev_copied, 0));
                if (sc.tri_tangents) kb_tangent_flag<<<g_n, 256, 0, st>>>(A);
                attrs_joined = true;
            }
            if (int rc = fetch_counters()) return rc;
            if (hc.n_active[level & 1] == 0) break;
        }
        kb_bin<<<g_n, 256, 0, st>>>(A, level, parity);
        kb_split<<<g_split, 128, 0, st>>>(A, level);
        kb_flags<<<g_n, 256, 0, st>>>(A, level, parity);
        kb_scan<<<1, 1024, 0, st>>>(A.words, A.wscan, n_bin_words, nullptr, &A.c->n_active[level & 1]);
        kb_scatter<<<g_n, 256, 0, st>>>(A, level, parity);
        parity ^= 1;
        if (timing && level < 6) lap(("L" + std::to_string(level)).c_str());
    }
    lap("big");
    CU_CHECK(cudaGetLastError());
    const bool with_tangents = sc.tri_tangents && hc.any_tangent;
    if (with_tangents) {
        if (int rc = d.tangents.alloc(n)) return rc;
        A.tangents = d.tangents.p;
    }
    if (hc.n_small) kb_small<<<(hc.n_small + 3) / 4, 128, 0, st>>>(A, parity);
    lap("small");
    kb_tris<<<(n + 1 + 255) / 256, 256, 0, st>>>(A, parity, with_tangents ? 1 : 0);
    lap("tris");
    kb_mark_root<<<1, 1, 0, st>>>(A);
    if (int rc = fetch_counters()) return rc;  // max_depth now covers kb_small's sub-trees
    for (uint32_t l = 0; l <= hc.max_depth; ++l)  // a wide level consumes at least one binary level
        kb_mark<<<256, 128, 0, st>>>(A, l);
    lap("mark");
    const uint32_t ns32 = static_cast<uint32_t>(n_slots);
    kb_markwords<<<(ns32 + 255) / 256, 256, 0, st>>>(A, ns32);
    kb_scan<<<1, 1024, 0, st>>>(A.words, A.wscan, (ns32 + 31) / 32, &A.c->n_wide, nullptr);
    kb_emit<<<(ns32 + 127) / 128, 128, 0, st>>>(A, ns32);
    CU_CHECK(cudaGetLastError());
    if (int rc = fetch_counters()) return rc;
    lap("emit");
    if (timing) std::fprintf(stderr, "rt_gpu device build phases (ms, serialised):%s\n", phases.c_str());
    d.built = A;
    d.built_parity = parity;
    d.built_info[1] = ns32;
    d.built_info[2] = hc.n_wide;
    d.built_info[3] = hc.n_wide ? 0u : static_cast<uint32_t>(~0);  // root link: wide node 0, or the single leaf at triangle 0
    d.built_info[4] = hc.stack_need;
    d.built_info[5] = hc.max_depth;
    d.built_info[7] = level;
    if (hc.error) return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: non-finite triangle or a node that cannot be quantised");
    if (hc.stack_need > RT_EXT_STACK_CAP) return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: the 4-wide tree needs more than RT_EXT_STACK_CAP traversal-stack entries");
    return RT_OK;
}

// The light side of a packed scene on device d (light nodes, light triangles, the sampling list, DLight records, the
// light box) and the DScene fields that refer to it.  Shared by rt_gpu_upload_scene and rt_gpu_update_geometry.
int upload_lights(DeviceState &d, const rt::PackedScene &p, uint32_t n_lights) {
#if RT_EXT_WIDE8  // only the node format the traversal kernel was built for goes to the device
    if (int rc = d.lqnodes8.upload(p.light.qnodes8, d.stream)) return rc;
#else
    if (int rc = d.lqnodes4.upload(p.light.qnodes4, d.stream)) return rc;
#endif
    {   // box of all light triangles, widened by 1e-4 of its size and of the coordinates' magnitude: a ray that misses
        // it has no light-pdf term (k_lightpdf); the last entry of light.tris is the null triangle
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        const size_t n_lt = p.light.tris.empty() ? 0 : p.light.tris.size() - 1;
        for (size_t k = 0; k < n_lt; ++k) {
            const DTri &t = p.light.tris[k];
            const float v[3][3] = {{t.ax, t.ay, t.az}, {t.ax + t.e1x, t.ay + t.e1y, t.az + t.e1z}, {t.ax + t.e2x, t.ay + t.e2y, t.az + t.e2z}};
            for (int j = 0; j < 3; ++j)
                for (int a = 0; a < 3; ++a) {
                    lo[a] = std::min(lo[a], v[j][a]);
                    hi[a] = std::max(hi[a], v[j][a]);
                }
        }
        for (int a = 0; a < 3; ++a) {
            const float m = n_lt ? 1e-4f * std::max({hi[a] - lo[a], std::fabs(lo[a]), std::fabs(hi[a]), 1e-3f}) : 0.0f;
            d.light_box.lo[a] = lo[a] - m;
            d.light_box.hi[a] = hi[a] + m;
        }
    }
    if (int rc = d.ltris.upload(p.light.tris, d.stream)) return rc;
    if (int rc = d.lsample.upload(p.light_sample, d.stream)) return rc;
    if (int rc = d.light_extra.upload(p.light_extra, d.stream)) return rc;
    d.scene.light.root4 = p.light.root4;
    d.scene.light.n_nodes8 = static_cast<uint32_t>(p.light.qnodes8.size());
    d.scene.light.root = p.light.root;
    d.scene.light.n_tris = static_cast<uint32_t>(p.light.tris.size());
    d.scene.n_lights = n_lights;
    d.scene.light.qnodes4 = d.lqnodes4.p;
    d.scene.light.qnodes8 = d.lqnodes8.p;
    d.scene.light.nodes = nullptr;
    d.scene.light.qnodes = nullptr;
    d.scene.light.tris = d.ltris.p;
    d.scene.light_sample = d.lsample.p;
    d.scene.light_extra = d.light_extra.p;
    return RT_OK;
}

// The node halves k_extend reads: [scene lo | light lo | scene hi | light hi], 32 bytes per node and half.  Its layout
// depends on both node counts, so an update of the light BVH makes it again.
int split_nodes(DeviceState &d, size_t n_scene, size_t n_light) {
#if !RT_EXT_WIDE8
    const size_t n_all = std::max<size_t>(n_scene + n_light, 1);
    if (int rc = d.q4split.alloc(n_all * 4)) return rc;
    char *lo = reinterpret_cast<char *>(d.q4split.p), *hi = lo + n_all * 32;
    if (n_scene) rt::k_split_nodes<<<static_cast<uint32_t>((n_scene * 4 + 255) / 256), 256, 0, d.stream>>>(d.qnodes4.p, static_cast<uint32_t>(n_scene), lo, hi);
    if (n_light) rt::k_split_nodes<<<static_cast<uint32_t>((n_light * 4 + 255) / 256), 256, 0, d.stream>>>(d.lqnodes4.p, static_cast<uint32_t>(n_light), lo + n_scene * 32, hi + n_scene * 32);
    CU_CHECK(cudaGetLastError());
    d.scene.scene.q4lo = lo;
    d.scene.light.q4lo = lo + n_scene * 32;
    d.scene.scene.q4_hi_off = d.scene.light.q4_hi_off = static_cast<uint32_t>(n_all * 32);
#else
    (void)d, (void)n_scene, (void)n_light;
#endif
    return RT_OK;
}

// rt_gpu_update_geometry on one device: the new positions, normals and tangents go into the build's input copies, the
// binary boxes are refit from the leaves up, the 4-wide nodes re-quantised and DTri / DAttr (/ DTangent) rewritten.  The
// topology stays the upload's (gpu_build.cuh, "refit").  `phases`: RT_TIMING's serialised phase times.
int device_refit_scene(DeviceState &d, const rt_geometry_update &u, std::string &phases) {
    using namespace rtb;
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t n = d.built_info[0], n_slots = d.built_info[1], n_wide = d.built_info[2], depth = d.built_info[5];
    const int parity = d.built_parity;
    cudaStream_t st = d.stream;
    Arrays A = d.built;
    Counters &hc = *d.h_counters;
    auto fetch_counters = [&]() -> int {
        CU_CHECK(cudaMemcpyAsync(&hc, A.c, sizeof(Counters), cudaMemcpyDeviceToHost, st));
        CU_CHECK(cudaStreamSynchronize(st));
        return RT_OK;
    };
    const bool timing = std::getenv("RT_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char *name) {
        if (!timing) return;
        cudaStreamSynchronize(st);
        const auto now = std::chrono::steady_clock::now();
        char buf[64];
        std::snprintf(buf, sizeof buf, " %s %.3f", name, std::chrono::duration<double, std::milli>(now - t_last).count());
        phases += buf;
        t_last = now;
    };
    if (n == 0) return RT_OK;  // only the null triangle
    if (!d.refit_ready) {  // from the pristine tree, before any box changes
        size_t off = 0;
        auto carve = [&](size_t bytes) {
            const size_t at = off;
            off += (bytes + 255) / 256 * 256;
            return at;
        };
        const size_t o_order = carve(static_cast<size_t>(n_slots) * 4), o_lstart = carve(kMaxLevels * 4), o_lcount = carve(kMaxLevels * 4);
        const size_t o_wslot = carve(std::max<size_t>(n_wide, 1) * 16);
        if (int rc = d.refit_scratch.alloc(off)) return rc;
        uint8_t *base = d.refit_scratch.p;
        Refit &R = d.refit;
        R.order = reinterpret_cast<uint32_t *>(base + o_order);
        R.lstart = reinterpret_cast<uint32_t *>(base + o_lstart);
        R.lcount = reinterpret_cast<uint32_t *>(base + o_lcount);
        R.wslot = reinterpret_cast<int32_t *>(base + o_wslot);
        CU_CHECK(cudaMemsetAsync(R.lcount, 0, kMaxLevels * 4, st));
        kr_levels_init<<<1, 1, 0, st>>>(R);
        const uint32_t g = std::min<uint32_t>((n + 255) / 256, 1024);
        for (uint32_t l = 0; l < depth; ++l) kr_levels<<<g, 256, 0, st>>>(A, R, l);
        if (n_wide) kr_wide_slots<<<(n_slots + 127) / 128, 128, 0, st>>>(A, R, n_slots);
        CU_CHECK(cudaGetLastError());
        d.refit_lstart.resize(depth + 1);
        d.refit_lcount.resize(depth + 1);
        CU_CHECK(cudaMemcpyAsync(d.refit_lstart.data(), R.lstart, (depth + 1) * 4, cudaMemcpyDeviceToHost, st));
        CU_CHECK(cudaMemcpyAsync(d.refit_lcount.data(), R.lcount, (depth + 1) * 4, cudaMemcpyDeviceToHost, st));
        if (int rc = fetch_counters()) return rc;
        if (hc.error) return fail(RT_ERR_CUDA, "rt_gpu_update_geometry: the recorded 4-wide grouping does not reproduce the uploaded links");
        d.refit_ready = true;
        lap("record");
    }
    CU_CHECK(cudaMemcpyAsync(d.in_pos.p, u.tri_pos, static_cast<size_t>(n) * 36, cudaMemcpyHostToDevice, st));
    CU_CHECK(cudaMemcpyAsync(d.in_nrm.p, u.tri_normals, static_cast<size_t>(n) * 36, cudaMemcpyHostToDevice, st));
    if (u.tri_tangents) {
        if (int rc = d.in_tan.alloc(static_cast<size_t>(n) * 9)) return rc;
        CU_CHECK(cudaMemcpyAsync(d.in_tan.p, u.tri_tangents, static_cast<size_t>(n) * 36, cudaMemcpyHostToDevice, st));
    }
    A.tri_tangents = u.tri_tangents ? d.in_tan.p : nullptr;
    lap("h2d");
    CU_CHECK(cudaMemsetAsync(&A.c->error, 0, 2 * sizeof(uint32_t), st));  // error, any_tangent
    if (A.tri_tangents) kb_tangent_flag<<<(n + 255) / 256, 256, 0, st>>>(A);
    for (uint32_t l = depth + 1; l-- > 0;)  // every level up to `depth` holds nodes
        kr_refit<<<(d.refit_lcount[l] + 255) / 256, 256, 0, st>>>(A, d.refit, d.refit_lstart[l], d.refit_lcount[l], parity);
    lap("refit");
    if (n_wide) kr_requant<<<(n_wide + 127) / 128, 128, 0, st>>>(A, d.refit, n_wide);
    CU_CHECK(cudaGetLastError());
    if (int rc = fetch_counters()) return rc;
    lap("quantise");
    if (hc.error) return fail(RT_ERR_BAD_SCENE, "rt_gpu_update_geometry: non-finite triangle or a node that cannot be quantised; the scene is gone");
    const bool with_tangents = A.tri_tangents && hc.any_tangent;
    A.tangents = nullptr;
    if (with_tangents) {
        if (int rc = d.tangents.alloc(n)) return rc;
        A.tangents = d.tangents.p;
    }
    kb_tris<<<(n + 1 + 255) / 256, 256, 0, st>>>(A, parity, with_tangents ? 1 : 0);
    CU_CHECK(cudaGetLastError());
    d.built = A;
    d.scene.tangents = A.tangents;
    lap("tris");
    return RT_OK;
}

// Structural check of a host BVH before anything is dereferenced through it; null when it is well formed
const char *bvh_problem(const rt_bvh_desc &b, uint32_t n_tris) {
    if (b.root != RT_NO_CHILD && b.root >= b.n_nodes) return "BVH root out of range";
    for (uint32_t i = 0; i < b.n_objects; ++i)
        if (b.objects[i] >= n_tris) return "BVH object id out of range";
    for (uint32_t i = 0; i < b.n_nodes; ++i) {
        const rt_bvh_node &nd = b.nodes[i];
        if ((nd.left_child != RT_NO_CHILD && nd.left_child >= b.n_nodes) || (nd.right_child != RT_NO_CHILD && nd.right_child >= b.n_nodes) ||
            nd.obj_begin > nd.obj_end || nd.obj_end > b.n_objects)
            return "BVH node links out of range";
    }
    return nullptr;
}

int upload_to_device(DeviceState &d, const rt_scene_desc &sc, const rt::PackedScene &p, bool device_built) {
    CU_CHECK(cudaSetDevice(d.device));
#if RT_EXT_WIDE8  // only the node format the traversal kernel was built for goes to the device
    if (int rc = d.qnodes8.upload(p.scene.qnodes8, d.stream)) return rc;
#else
    if (!device_built)
        if (int rc = d.qnodes4.upload(p.scene.qnodes4, d.stream)) return rc;
#endif
    if (!device_built) {
        if (int rc = d.tris.upload(p.scene.tris, d.stream)) return rc;
        if (int rc = d.attrs.upload(p.attrs, d.stream)) return rc;
        if (int rc = d.tangents.upload(p.tangents, d.stream)) return rc;
        std::memset(d.built_info, 0, sizeof d.built_info);
    }
    if (int rc = d.materials.upload(p.materials, d.stream)) return rc;
    if (int rc = d.textures.upload(p.textures, d.stream)) return rc;
    if (int rc = d.texels.upload(p.texels, d.stream)) return rc;
    std::vector<float> lut(p.gamma_lut, p.gamma_lut + 256);
    if (int rc = d.lut.upload(lut, d.stream)) return rc;
    rt::fill_scene_constants(sc, p, d.scene);
    if (int rc = upload_lights(d, p, sc.light_bvh.n_objects)) return rc;
    d.scene.scene.nodes = nullptr;  // the device traverses the quantised copies only
    d.scene.scene.qnodes = nullptr;  // the 2-wide form exists on the host only (tests)
    d.scene.scene.qnodes4 = d.qnodes4.p;
    d.scene.scene.qnodes8 = d.qnodes8.p;
    if (int rc = split_nodes(d, device_built ? d.built_info[2] : p.scene.qnodes4.size(), p.light.qnodes4.size())) return rc;
    d.scene.scene.tris = d.tris.p;
    d.scene.attrs = d.attrs.p;
    d.scene.tangents = p.tangents.empty() ? nullptr : d.tangents.p;
    if (device_built) {
        d.scene.scene.root4 = static_cast<int32_t>(d.built_info[3]);
        d.scene.scene.n_tris = d.built_info[0] + 1;
        d.scene.tangents = d.built.tangents;
    }
    d.scene.materials = d.materials.p;
    d.scene.textures = d.textures.p;
    d.scene.texels = d.texels.p;
    CU_CHECK(cudaStreamSynchronize(d.stream));
    return RT_OK;
}

rt::Camera make_camera(const rt_camera &s, uint32_t w, uint32_t h) {
    rt::Camera c;
    c.pos = rt::mk3(s.position[0], s.position[1], s.position[2]);
    c.right = rt::mk3(s.right[0], s.right[1], s.right[2]);
    c.up = rt::mk3(s.up[0], s.up[1], s.up[2]);
    c.fwd = rt::mk3(s.forward[0], s.forward[1], s.forward[2]);
    // tan(fov_x / 2) and Camera::fov_y (scene.h:69-71), evaluated on the host exactly like the reference
    c.tan_half_x = std::tan(s.fov_x / 2);
    const float fov_y = std::atan(std::tan(s.fov_x / 2) * static_cast<float>(h) / static_cast<float>(w)) * 2;
    c.tan_half_y = std::tan(fov_y / 2);
    c.inv_w2 = 2.0f / static_cast<float>(w);
    c.inv_h2 = 2.0f / static_cast<float>(h);
    return c;
}

// The camera of the uploaded triangle scene (rt_scene_desc.camera)
rt_camera scene_camera(const DScene &s) {
    rt_camera c;
    for (int k = 0; k < 3; ++k) {
        c.position[k] = s.cam_pos[k];
        c.right[k] = s.cam_right[k];
        c.up[k] = s.cam_up[k];
        c.forward[k] = s.cam_fwd[k];
    }
    c.fov_x = s.fov_x;
    return c;
}

// The cameras of a multi-view render (rt_gpu_render_views), one per view, and the Philox key of its first view.
// rt_gpu_render_projected adds one projection per view (projection.cuh); without them queue 0 is k_generate_views.
static_assert(sizeof(rt::Projection) == sizeof(rt_projection) && rt::kProjPinhole == RT_PROJ_PINHOLE && rt::kProjThinLens == RT_PROJ_THIN_LENS &&
                  rt::kProjOrthographic == RT_PROJ_ORTHOGRAPHIC && rt::kProjEquirect == RT_PROJ_EQUIRECT,
              "rt::Projection mirrors rt_projection");
struct ViewSet {
    std::vector<rt::Camera> cams;
    std::vector<rt::Projection> projs;
    uint32_t view_base = 0;
};

// Uploads the cameras of `views` (and their projections) to device d on its stream
int upload_views(DeviceState &d, const ViewSet &views) {
    if (int rc = d.cams.upload(views.cams, d.stream)) return rc;
    if (!views.projs.empty())
        if (int rc = d.projs.upload(views.projs, d.stream)) return rc;
    return RT_OK;
}

void mark(rt_gpu_ctx *ctx, DeviceState &d, int kind) {
    if (!ctx->profiling) return;
    cudaEvent_t e = d.next_event();
    cudaEventRecord(e, d.stream);
    d.marks.emplace_back(e, kind);
}

// Course text scene: one launch, one thread per pixel (text_kernels.cuh).
int enqueue_text_render(rt_gpu_ctx *ctx, DeviceState &d, int dev_index, const rt_render_params &rp, uint32_t s_begin, uint32_t s_end,
                        uint64_t &launches) {
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t W = rp.width, H = rp.height;
    const size_t n_pix = static_cast<size_t>(W) * H;
    if (int rc = d.accum.alloc(n_pix)) return rc;
    if (int rc = d.stats.alloc(4)) return rc;
    const bool ids_mode = rp.mode == RT_MODE_PRIMARY_IDS;
    if (ids_mode) {
        if (int rc = d.prim_ids.alloc(n_pix)) return rc;
    } else if (!(rp.flags & RT_FLAG_ACCUMULATE) || dev_index > 0) {  // see enqueue_render
        CU_CHECK(cudaMemsetAsync(d.accum.p, 0, n_pix * sizeof(float4), d.stream));
    }
    d.marks.clear();
    d.events_used = 0;
    CU_CHECK(cudaEventRecord(d.ev_begin, d.stream));
    mark(ctx, d, -1);
    const uint32_t px_begin = ids_mode ? 0u : rp.pixel_begin;
    const uint32_t px_end = ids_mode || rp.pixel_end == 0 ? static_cast<uint32_t>(n_pix) : rp.pixel_end;
    const uint32_t n_render = px_end > px_begin ? px_end - px_begin : 0u;
    const unsigned long long hs[4] = {0, 0, 0, ids_mode ? 0ull : static_cast<unsigned long long>(n_render) * (s_end - s_begin)};
    CU_CHECK(cudaMemcpyAsync(d.stats.p, hs, sizeof hs, cudaMemcpyHostToDevice, d.stream));
    if (n_render > 0 && (ids_mode || (s_end > s_begin && d.tscene.ray_depth > 0))) {
        const rt::Camera cam = make_camera(d.tcamera, W, H);
        rtt::TextParams tp;
        tp.width = W;
        tp.height = H;
        tp.s0 = s_begin;
        tp.s1 = s_end;
        tp.k0 = static_cast<uint32_t>(rp.seed);
        tp.k1 = static_cast<uint32_t>(rp.seed >> 32);
        tp.ids = ids_mode ? 1u : 0u;
        tp.pix0 = px_begin;
        tp.npix = n_render;
        rtt::k_text_render<<<(n_render + 127) / 128, 128, 0, d.stream>>>(d.tscene, cam, tp, d.accum.p, d.prim_ids.p);
        mark(ctx, d, K_SHADE);
        launches += 1;
    }
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
    return RT_OK;
}

// Paths in flight per batch.  Every kernel of a batch ends with a tail in which the last warps finish
// their rays while the other SMs idle, so throughput grows with the batch: 8 Mi / 16 / 32 / 64 / 128 /
// 256 Mi paths -> 771 / 819 / 845 / 881 / 896 / 910 Msamples/s on config 4 (B200, measured; a later build: 128 / 256 /
// 512 / 640 Mi -> 1149 / 1163 / 1169 / 1169).  The default is 512 Mi paths (140 B of queue state each = 75 GB of the
// 180 GB), capped at half of the free memory.
// bytes_per_path: what one path of the batch needs; held_paths / held_bytes: the paths the handle's buffers already hold
// and their bytes (given back to the free memory when they grow)
size_t batch_cap_of(uint32_t max_paths_in_flight, size_t want_total, size_t bytes_per_path, size_t held_paths, size_t held_bytes) {
    size_t max_paths = max_paths_in_flight;
    if (max_paths == 0) {
        max_paths = static_cast<size_t>(512) << 20;
        // the memory query is a slow, jittery driver call (tens of ms with 50 GB allocated): only when the queues
        // would have to grow beyond what this handle already holds
        if (std::min(max_paths, want_total) > held_paths) {
            size_t free_b = 0, total_b = 0;
            if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
                max_paths = std::min(max_paths, std::max(held_paths, (free_b + held_bytes) / 2 / bytes_per_path));
        }
    }
    max_paths = std::max<size_t>(max_paths, 1024);
    return std::min(max_paths, want_total);
}
size_t batch_cap(const DeviceState &d, uint32_t max_paths_in_flight, size_t want_total) {
    return batch_cap_of(max_paths_in_flight, want_total, kBytesPerPath, d.queue_cap, d.queue_cap * kBytesPerPath);
}

size_t n_counters_of(uint32_t qdepth) { return (6 * static_cast<size_t>(qdepth) + 2) * rt::kCounterStride; }  // one 256-byte line each

// Queues of bounce b: in = parity b & 1, out = the other one (k_generate fills queue 0 through `out` of b = -1)
rt::Queues queues_of(DeviceState &d, uint32_t qdepth, int b) {
    rt::Queues q;
    const int in = b & 1, out = in ^ 1;
    q.o_in = d.qo[in];
    q.d_in = d.qd[in];
    q.thr_in = d.qthr[in];
    q.o_out = d.qo[out];
    q.d_out = d.qd[out];
    q.thr_out = d.qthr[out];
    q.hit = d.hit;
    q.rad = d.rad;
    q.count = d.counters.p;
    q.fetch_ext = d.counters.p + (qdepth + 1) * rt::kCounterStride;
    q.fetch_shade = d.counters.p + (2 * qdepth + 1) * rt::kCounterStride;
    q.stats = d.stats.p;
    q.lpdf = d.lpdf[in];
    q.lpdf_out = d.lpdf[out];
    q.light_list = d.light_list;
    q.light_count = d.counters.p + (3 * qdepth + 1) * rt::kCounterStride;
    return q;
}

// The bounce loop of one batch whose queue 0 is filled (at most n paths): k_lightpdf_list / k_extend / k_shade per
// bounce.  On return every kernel of the batch is ordered before the next work on d.stream.
int enqueue_bounces(rt_gpu_ctx *ctx, DeviceState &d, const rt::BatchParams &bp, uint32_t n, bool split_allowed, uint64_t &launches) {
    const uint32_t depth = d.scene.ray_depth, qdepth = std::max(depth, 1u);
    const float inv_n_lights = d.scene.n_lights ? 1.0f / static_cast<float>(d.scene.n_lights) : 0.0f;
#if !RT_EXT_WIDE8
    // Batches below 256 Mi paths: two halves of every queue on two streams.  A persistent kernel ends with a drain
    // (once its queue is empty every warp runs on with fewer and fewer live lanes and the SMs empty out), a fixed
    // cost per launch.  With the halves in flight together the other half's next kernel moves into the freed
    // slots: E(b, 0) | E(b, 1) over E(b, 0)'s drain | S(b, 0) over E(b, 1)'s drain | S(b, 1) over S(b, 0)'s; only
    // the last shade of a bounce drains in the open (both halves of queue b + 1 need both shades of queue b).
    // Measured on config 4: 92.05 -> 91.07 ms at 125 spp (the 8-GPU share of the image), 709.7 -> 711.6 ms at
    // 1000 spp in 512 Mi-path batches, hence the bound.
    const bool split = split_allowed && n < (256u << 20);
    if (split) {
        cudaStream_t sa = d.stream, sb = d.stream2;
        CU_CHECK(cudaEventRecord(d.ev_a, sa));  // k_generate (and the counters' memset) done
        CU_CHECK(cudaStreamWaitEvent(sb, d.ev_a, 0));
        for (uint32_t b = 0; b < depth; ++b) {
            rt::Queues q0 = queues_of(d, qdepth, static_cast<int>(b)), q1 = q0;
            q1.fetch_ext = d.counters.p + (4 * qdepth + 2) * rt::kCounterStride;
            q1.fetch_shade = d.counters.p + (5 * qdepth + 2) * rt::kCounterStride;
            if (b > 0) {  // queue b is complete when both shades of queue b - 1 are
                CU_CHECK(cudaStreamWaitEvent(sa, d.ev_b, 0));
                CU_CHECK(cudaStreamWaitEvent(sb, d.ev_a, 0));
            }
            const bool light = RT_LIGHT_KERNEL && b > 0 && d.scene.n_lights > 0;
            if (light) {
                rt::k_lightpdf_list<<<d.light_blocks, rt::kLightThreads, 0, sa>>>(d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q0, b, 0x3F800000u);
                CU_CHECK(cudaEventRecord(d.ev_light, sa));
                ++launches;
            }
            rt::k_extend<<<d.extend_blocks, rt::kExtendThreads, 0, sa>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q0, b | rt::kPartFirst, 0x3F800000u);
            rt::k_extend<<<d.extend_blocks, rt::kExtendThreads, 0, sb>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q1, b | rt::kPartSecond, 0x3F800000u);
            rt::k_shade<<<d.shade_blocks, rt::kShadeThreads, 0, sa>>>(d.scene, d.lut.p, bp, q0, b | rt::kPartFirst, d.light_box);
            if (light) CU_CHECK(cudaStreamWaitEvent(sb, d.ev_light, 0));  // the light pdfs of queue b
            rt::k_shade<<<d.shade_blocks, rt::kShadeThreads, 0, sb>>>(d.scene, d.lut.p, bp, q1, b | rt::kPartSecond, d.light_box);
            CU_CHECK(cudaEventRecord(d.ev_a, sa));
            CU_CHECK(cudaEventRecord(d.ev_b, sb));
        }
        CU_CHECK(cudaStreamWaitEvent(sa, d.ev_b, 0));
        launches += 4 * static_cast<uint64_t>(depth);
        return RT_OK;
    }
#else
    (void)split_allowed;
    (void)n;
#endif
    for (uint32_t b = 0; b < depth; ++b) {
        const rt::Queues q = queues_of(d, qdepth, static_cast<int>(b));
#if RT_LIGHT_KERNEL
        if (b > 0 && d.scene.n_lights > 0) {  // queue 0 holds camera rays: nothing is pending
            rt::k_lightpdf_list<<<d.light_blocks, rt::kLightThreads, 0, d.stream>>>(d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q, b, 0x3F800000u);
            mark(ctx, d, K_LIGHTPDF);
            ++launches;
        }
#endif
        RT_K_EXTEND<<<d.extend_blocks, rt::kExtendThreads, 0, d.stream>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q, b, 0x3F800000u);
        mark(ctx, d, K_EXTEND);
        rt::k_shade<<<d.shade_blocks, rt::kShadeThreads, 0, d.stream>>>(d.scene, d.lut.p, bp, q, b, d.light_box);
        mark(ctx, d, K_SHADE);
    }
    launches += 2 * static_cast<uint64_t>(depth);
    return RT_OK;
}

// Enqueue the whole render of samples [s_begin, s_end) on device d (asynchronous).  views != nullptr: the stacked image
// of its views (views.cuh), rp's pixel range indexing it.
int enqueue_render(rt_gpu_ctx *ctx, DeviceState &d, int dev_index, const rt_render_params &rp, uint32_t s_begin, uint32_t s_end,
                   const ViewSet *views, uint64_t &launches) {
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t W = rp.width, H = rp.height, depth = d.scene.ray_depth;
    const uint32_t n_views = views ? static_cast<uint32_t>(views->cams.size()) : 1u;
    const size_t n_pix = static_cast<size_t>(W) * H * n_views;
    const rt::Camera cam = make_camera(scene_camera(d.scene), W, H);
    // stacked pixel + key_offset = Philox pixel key; fits 32 bits (rt_gpu_render_views checks (view_base + V) * W * H)
    const uint32_t key_offset = views ? static_cast<uint32_t>(static_cast<uint64_t>(views->view_base) * W * H) : 0u;
    if (int rc = d.accum.alloc(n_pix)) return rc;
    if (int rc = d.stats.alloc(4)) return rc;
    CU_CHECK(cudaMemsetAsync(d.stats.p, 0, 4 * sizeof(unsigned long long), d.stream));
    const bool ids_mode = rp.mode == RT_MODE_PRIMARY_IDS;
    // RT_FLAG_ACCUMULATE keeps the sums of device 0 only: the reduce leaves the total there, while devices 1..n-1
    // still hold their partial sums of the previous render, which the next reduce would add a second time
    if (!ids_mode && (!(rp.flags & RT_FLAG_ACCUMULATE) || dev_index > 0))
        CU_CHECK(cudaMemsetAsync(d.accum.p, 0, n_pix * sizeof(float4), d.stream));
    d.marks.clear();
    d.events_used = 0;
    CU_CHECK(cudaEventRecord(d.ev_begin, d.stream));
    mark(ctx, d, -1);

    if (!ids_mode && (s_end <= s_begin || depth == 0 || (rp.pixel_end != 0 && rp.pixel_end <= rp.pixel_begin))) {  // run_raytracer returns early for ray_depth == 0, raytracer.h:630
        CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
        return RT_OK;
    }

    if (ids_mode) {
        if (int rc = d.prim_ids.alloc(n_pix)) return rc;
        s_begin = 0;
        s_end = 1;
    }
    const size_t px_begin = ids_mode ? 0 : rp.pixel_begin, px_end = ids_mode || rp.pixel_end == 0 ? n_pix : rp.pixel_end;
    const size_t n_render = px_end - px_begin;  // image-tile split: only this pixel range is rendered
    const size_t cap = batch_cap(d, rp.max_paths_in_flight, n_render * static_cast<size_t>(s_end - s_begin));
    if (int rc = d.alloc_queues(cap)) return rc;
    const uint32_t qdepth = std::max(depth, 1u);
    const size_t n_counters = n_counters_of(qdepth);
    if (int rc = d.counters.alloc(n_counters)) return rc;
    const rt::Queues q_gen = queues_of(d, qdepth, -1);
    if (views)
        if (int rc = upload_views(d, *views)) return rc;
    // per-kernel profiling needs the kernels one after the other on one stream
    const bool split_allowed = !ids_mode && !ctx->profiling && !std::getenv("RT_NO_SPLIT");

    const float inv_n_lights = d.scene.n_lights ? 1.0f / static_cast<float>(d.scene.n_lights) : 0.0f;
    rt::BatchParams bp;
    bp.width = W;
    bp.height = H;
    bp.k0 = static_cast<uint32_t>(rp.seed);
    bp.k1 = static_cast<uint32_t>(rp.seed >> 32);
    bp.centre = ids_mode ? 1u : 0u;

    // batches: all pixels x k samples when the image fits, else pixel chunks x 1 sample
    const size_t pix_chunk = std::max<size_t>(1, std::min(n_render, cap));
    for (size_t pix0 = px_begin; pix0 < px_end; pix0 += pix_chunk) {
        const uint32_t npix = static_cast<uint32_t>(std::min(pix_chunk, px_end - pix0));
        const uint32_t k_max = static_cast<uint32_t>(std::max<size_t>(1, cap / npix));
        for (uint32_t s0 = s_begin; s0 < s_end; s0 += k_max) {
            bp.pix0 = static_cast<uint32_t>(pix0);
            bp.npix = npix;
            bp.s0 = s0;
            bp.k = std::min(k_max, s_end - s0);
            bp.tiled = !ids_mode && pix0 == 0 && npix == n_pix && W % 8 == 0 && (H * n_views) % 4 == 0 && !std::getenv("RT_NO_TILES");
            const uint32_t n = bp.npix * bp.k;
            CU_CHECK(cudaMemsetAsync(d.counters.p, 0, n_counters * sizeof(uint32_t), d.stream));
            if (views && !views->projs.empty())
                rt::k_generate_proj<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, d.projs.p, bp, q_gen, key_offset);
            else if (views)
                rt::k_generate_views<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, bp, q_gen, key_offset);
            else
                rt::k_generate<<<(n + 255) / 256, 256, 0, d.stream>>>(cam, bp, q_gen);
            mark(ctx, d, K_GENERATE);
            if (ids_mode) {  // pixel-centre rays through the same traversal kernel, then hit -> scene.objects id
                RT_K_EXTEND<<<d.extend_blocks, rt::kExtendThreads, 0, d.stream>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, queues_of(d, qdepth, 0), 0, 0x3F800000u);
                mark(ctx, d, K_EXTEND);
                rt::k_ids_from_hits<<<(bp.npix + 255) / 256, 256, 0, d.stream>>>(bp, d.hit, d.scene.scene.tris, d.prim_ids.p);
                mark(ctx, d, K_IDS);
                launches += 3;
                continue;
            }
            rt::BatchParams bp_key = bp;  // k_shade's radiance slot: (sample - s0) * npix + (key - pix0)
            bp_key.pix0 += key_offset;
            if (int rc = enqueue_bounces(ctx, d, bp_key, n, split_allowed, launches)) return rc;
            rt::k_accumulate<<<(bp.npix + 255) / 256, 256, 0, d.stream>>>(bp, d.rad, d.accum.p);
            mark(ctx, d, K_ACCUMULATE);
            launches += 2;
        }
    }
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
    return RT_OK;
}

// Enqueue the AOV render (aov.cuh) of samples [0, samples) on device d: enqueue_render's batches and queue 0, then per
// bounce k_extend and k_aov_step, then k_aov_accumulate into d.aov_sums.  RT_MODE_PRIMARY_IDS: the pixel-centre rays of
// that mode (sample 0, the whole image).  Touches none of the beauty render's sums, counts, ids or stats.
int enqueue_render_aov(DeviceState &d, const rt_render_params &rp, const ViewSet *views, uint64_t &launches) {
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t W = rp.width, H = rp.height, depth = d.scene.ray_depth;
    const uint32_t n_views = views ? static_cast<uint32_t>(views->cams.size()) : 1u;
    const size_t n_pix = static_cast<size_t>(W) * H * n_views;
    const rt::Camera cam = make_camera(scene_camera(d.scene), W, H);
    const uint32_t key_offset = views ? static_cast<uint32_t>(static_cast<uint64_t>(views->view_base) * W * H) : 0u;
    const bool centre = rp.mode == RT_MODE_PRIMARY_IDS;
    if (int rc = d.aov_sums.alloc(3 * n_pix)) return rc;
    if (int rc = d.stats.alloc(4)) return rc;
    CU_CHECK(cudaMemsetAsync(d.stats.p, 0, 4 * sizeof(unsigned long long), d.stream));
    CU_CHECK(cudaMemsetAsync(d.aov_sums.p, 0, 3 * n_pix * sizeof(float4), d.stream));
    const rt::AovPlanes sums{d.aov_sums.p, d.aov_sums.p + n_pix, d.aov_sums.p + 2 * n_pix};
    CU_CHECK(cudaEventRecord(d.ev_begin, d.stream));
    const uint32_t s_end = centre ? 1u : rp.samples;
    const size_t px_begin = centre ? 0 : rp.pixel_begin, px_end = centre ? n_pix : rp.pixel_end;
    const size_t n_render = px_end - px_begin;
    if (depth == 0 || n_render == 0) {  // no hit is walked: every value is 0
        CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
        return RT_OK;
    }
    const size_t cap = batch_cap_of(rp.max_paths_in_flight, n_render * static_cast<size_t>(s_end), kBytesPerPath + kAovBytesPerPath,
                                    std::min(d.queue_cap, d.aov_cap), d.queue_cap * kBytesPerPath + d.aov_cap * kAovBytesPerPath);
    if (int rc = d.alloc_queues(cap)) return rc;
    if (cap > d.aov_cap) {
        d.aov_cap = 0;
        if (int rc = d.aov_slots.alloc(3 * cap)) return rc;
        d.aov_cap = cap;
    }
    const rt::AovPlanes slots{d.aov_slots.p, d.aov_slots.p + d.aov_cap, d.aov_slots.p + 2 * d.aov_cap};
    const uint32_t qdepth = std::max(depth, 1u);
    const size_t n_counters = n_counters_of(qdepth);
    if (int rc = d.counters.alloc(n_counters)) return rc;
    const rt::Queues q_gen = queues_of(d, qdepth, -1);
    if (views)
        if (int rc = upload_views(d, *views)) return rc;
    const float inv_n_lights = d.scene.n_lights ? 1.0f / static_cast<float>(d.scene.n_lights) : 0.0f;
    rt::BatchParams bp;
    bp.width = W;
    bp.height = H;
    bp.k0 = static_cast<uint32_t>(rp.seed);
    bp.k1 = static_cast<uint32_t>(rp.seed >> 32);
    bp.centre = centre ? 1u : 0u;
    // enqueue_render's batches: all pixels x k samples when the image fits, else pixel chunks x 1 sample
    const size_t pix_chunk = std::max<size_t>(1, std::min(n_render, cap));
    for (size_t pix0 = px_begin; pix0 < px_end; pix0 += pix_chunk) {
        const uint32_t npix = static_cast<uint32_t>(std::min(pix_chunk, px_end - pix0));
        const uint32_t k_max = static_cast<uint32_t>(std::max<size_t>(1, cap / npix));
        for (uint32_t s0 = 0; s0 < s_end; s0 += k_max) {
            bp.pix0 = static_cast<uint32_t>(pix0);
            bp.npix = npix;
            bp.s0 = s0;
            bp.k = std::min(k_max, s_end - s0);
            bp.tiled = !centre && pix0 == 0 && npix == n_pix && W % 8 == 0 && (H * n_views) % 4 == 0 && !std::getenv("RT_NO_TILES");
            const uint32_t n = bp.npix * bp.k;
            CU_CHECK(cudaMemsetAsync(d.counters.p, 0, n_counters * sizeof(uint32_t), d.stream));
            if (views && !views->projs.empty())
                rt::k_generate_proj<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, d.projs.p, bp, q_gen, key_offset);
            else if (views)
                rt::k_generate_views<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, bp, q_gen, key_offset);
            else
                rt::k_generate<<<(n + 255) / 256, 256, 0, d.stream>>>(cam, bp, q_gen);
            rt::BatchParams bp_key = bp;  // the slot of a path: (sample - s0) * npix + (key - pix0), as k_shade's
            bp_key.pix0 += key_offset;
            // the queues shrink with every bounce; their sizes live on the device, so every bounce is launched
            const uint32_t step_blocks = static_cast<uint32_t>(std::min<size_t>((n + rt::kAovThreads - 1) / rt::kAovThreads,
                                                                                static_cast<size_t>(d.sm_count) * 16));
            for (uint32_t b = 0; b < depth; ++b) {
                const rt::Queues q = queues_of(d, qdepth, static_cast<int>(b));
                RT_K_EXTEND<<<d.extend_blocks, rt::kExtendThreads, 0, d.stream>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q, b, 0x3F800000u);
                rt::k_aov_step<<<step_blocks, rt::kAovThreads, 0, d.stream>>>(d.scene, d.lut.p, bp_key, q, b, slots);
            }
            rt::k_aov_accumulate<<<(bp.npix + 255) / 256, 256, 0, d.stream>>>(bp, slots, sums);
            launches += 2 + 2 * static_cast<uint64_t>(depth);
        }
    }
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
    return RT_OK;
}

// One device's part of an adaptive render (rt_gpu_render_adaptive, rt_gpu_render_views_adaptive): the pixel range it
// adapts and where its rounds are.
struct AdaptiveRun {
    DeviceState *d = nullptr;
    size_t pix0 = 0, n_render = 0;
    uint32_t k_max = 0, n_words = 0, done = 0;  // samples per pixel and batch; flag words; samples every active pixel has
    int cur = 0;                                 // the list of the active pixels: alist + cur * n_render
    bool finished = false;
    rt::BatchParams bp{};
    rt::Camera cam{};
    uint32_t key_offset = 0;  // views: stacked pixel + key_offset = Philox pixel key (view_base * W * H)
};

// Sizes the queues and the adaptive buffers of run.d for the pixel range [pix0, pix1) and clears its sums, counts and
// errors; no kernel runs yet.  RT_ERR_INVALID_ARG when the range does not fit one batch at one sample.  views != nullptr:
// the stacked image of its views (views.cuh), [pix0, pix1) indexing it, and its cameras go to d.cams.
int setup_adaptive(rt_gpu_ctx *ctx, AdaptiveRun &run, const rt_render_params &rp, size_t pix0, size_t pix1, const ViewSet *views) {
    DeviceState &d = *run.d;
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t n_views = views ? static_cast<uint32_t>(views->cams.size()) : 1u;
    const size_t n_pix = static_cast<size_t>(rp.width) * rp.height * n_views;
    run.pix0 = pix0;
    run.n_render = pix1 - pix0;
    const size_t cap = batch_cap(d, rp.max_paths_in_flight, std::max<size_t>(run.n_render, 1) * rp.samples);
    if (run.n_render > cap)
        return fail(RT_ERR_INVALID_ARG, std::string(views ? "rt_gpu_render_views_adaptive" : "rt_gpu_render_adaptive") +
                                            ": the pixel range (" + std::to_string(run.n_render) + " pixels) does not fit one batch of " +
                                            std::to_string(cap) + " paths");
    run.k_max = static_cast<uint32_t>(cap / std::max<size_t>(run.n_render, 1));
    run.n_words = static_cast<uint32_t>((run.n_render + 31) / 32);
    run.cur = 0;
    run.done = 0;
    run.finished = run.n_render == 0 || d.scene.ray_depth == 0;  // run_raytracer returns early for ray_depth == 0
    if (int rc = d.accum.alloc(n_pix)) return rc;
    if (int rc = d.stats.alloc(4)) return rc;
    if (int rc = d.acounts.alloc(n_pix)) return rc;
    if (int rc = d.aerr.alloc(n_pix)) return rc;
    if (int rc = d.actr.alloc(2)) return rc;
    if (!run.finished) {
        if (int rc = d.alloc_queues(cap)) return rc;
        if (int rc = d.counters.alloc(n_counters_of(std::max(d.scene.ray_depth, 1u)))) return rc;
        if (int rc = d.alist.alloc(2 * run.n_render)) return rc;
        if (int rc = d.awords.alloc(2 * static_cast<size_t>(run.n_words))) return rc;
    }
    if (views)
        if (int rc = upload_views(d, *views)) return rc;
    d.apix0 = pix0;
    d.apix1 = pix1;
    CU_CHECK(cudaMemsetAsync(d.stats.p, 0, 4 * sizeof(unsigned long long), d.stream));
    CU_CHECK(cudaMemsetAsync(d.accum.p, 0, n_pix * sizeof(float4), d.stream));
    CU_CHECK(cudaMemsetAsync(d.acounts.p, 0, n_pix * sizeof(uint32_t), d.stream));
    CU_CHECK(cudaMemsetAsync(d.aerr.p, 0, n_pix * sizeof(float), d.stream));
    CU_CHECK(cudaMemsetAsync(d.actr.p, 0, 2 * sizeof(uint32_t), d.stream));
    rt::BatchParams &bp = run.bp;
    bp.pix0 = static_cast<uint32_t>(pix0);
    bp.npix = static_cast<uint32_t>(run.n_render);  // the whole range: k_shade's radiance slots stay those of a fixed render
    bp.width = rp.width;
    bp.height = rp.height;  // views: the height of one view (split_view_pixel)
    bp.k0 = static_cast<uint32_t>(rp.seed);
    bp.k1 = static_cast<uint32_t>(rp.seed >> 32);
    bp.centre = 0;
    bp.tiled = 0;  // queue 0 follows the active list, whose first form is already in tiles where that applies
    run.cam = make_camera(scene_camera(d.scene), rp.width, rp.height);
    // fits 32 bits: rt_gpu_render_views_adaptive checks (view_base + V) * W * H
    run.key_offset = views ? static_cast<uint32_t>(static_cast<uint64_t>(views->view_base) * rp.width * rp.height) : 0u;
    d.marks.clear();
    d.events_used = 0;
    CU_CHECK(cudaEventRecord(d.ev_begin, d.stream));
    mark(ctx, d, -1);
    return RT_OK;
}

// Round `round` of run.d (k samples for every pixel of the active list), asynchronous: batches of k_max samples, then
// the rule, the flag scan and the compaction into the other list, whose device-side length goes to h_active[round & 1]
// behind ev_round[round & 1].
int enqueue_adaptive_round(rt_gpu_ctx *ctx, AdaptiveRun &run, const rt_render_params &rp, const rt_adaptive_params &ap, uint32_t round,
                           uint32_t k, const ViewSet *views, uint64_t &launches) {
    DeviceState &d = *run.d;
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t qdepth = std::max(d.scene.ray_depth, 1u), npix = run.bp.npix;
    uint32_t *list = d.alist.p + run.cur * run.n_render, *next = d.alist.p + (run.cur ^ 1) * run.n_render;
    uint32_t *active = d.actr.p + run.cur, *next_active = d.actr.p + (run.cur ^ 1);
    uint32_t *words = d.awords.p, *wscan = d.awords.p + run.n_words;
    if (round == 0) {  // tiles over the stacked image of W x (V * H), as in k_generate_views
        const uint32_t n_views = views ? static_cast<uint32_t>(views->cams.size()) : 1u;
        const bool tiled = run.pix0 == 0 && npix == static_cast<size_t>(rp.width) * rp.height * n_views && rp.width % 8 == 0 &&
                           (rp.height * n_views) % 4 == 0 && !std::getenv("RT_NO_TILES");
        rt::k_adapt_init<<<(npix + 255) / 256, 256, 0, d.stream>>>(list, run.bp.pix0, npix, rp.width, tiled ? 1u : 0u, active);
        ++launches;
    }
    const rt::Queues q_gen = queues_of(d, qdepth, -1);
    const bool split_allowed = !ctx->profiling && !std::getenv("RT_NO_SPLIT");
    for (uint32_t j0 = 0; j0 < k; j0 += run.k_max) {
        rt::BatchParams bp = run.bp;
        bp.s0 = run.done + j0;
        bp.k = std::min(run.k_max, k - j0);
        const uint32_t n = npix * bp.k;  // the grid of k_generate_active; the queue holds n_active * k paths
        CU_CHECK(cudaMemsetAsync(d.counters.p, 0, n_counters_of(qdepth) * sizeof(uint32_t), d.stream));
        if (views && !views->projs.empty())
            rt::k_generate_active_proj<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, d.projs.p, bp, q_gen, list, active, run.key_offset);
        else if (views)
            rt::k_generate_active_views<<<(n + 255) / 256, 256, 0, d.stream>>>(d.cams.p, bp, q_gen, list, active, run.key_offset);
        else
            rt::k_generate_active<<<(n + 255) / 256, 256, 0, d.stream>>>(run.cam, bp, q_gen, list, active);
        mark(ctx, d, K_GENERATE);
        rt::BatchParams bp_key = bp;  // k_shade's radiance slot: (sample - s0) * npix + (key - pix0)
        bp_key.pix0 += run.key_offset;
        if (int rc = enqueue_bounces(ctx, d, bp_key, n, split_allowed, launches)) return rc;
        rt::k_accumulate_active<<<(npix + 255) / 256, 256, 0, d.stream>>>(bp, d.rad, d.accum.p, d.acounts.p, list, active);
        mark(ctx, d, K_ACCUMULATE);
        launches += 2;
    }
    run.done += k;
    rt::k_adapt_flags<<<(run.n_words * 32 + 255) / 256, 256, 0, d.stream>>>(list, active, d.accum.p, d.acounts.p, d.aerr.p, rp.samples,
                                                                               ap.rel_error, ap.abs_floor, words, run.n_words);
    rtb::kb_scan<<<1, 1024, 0, d.stream>>>(words, wscan, run.n_words, next_active, nullptr);
    rt::k_adapt_scatter<<<(npix + 255) / 256, 256, 0, d.stream>>>(list, next, active, words, wscan);
    launches += 3;
    CU_CHECK(cudaMemcpyAsync(d.h_active + (round & 1), next_active, sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaEventRecord(d.ev_round[round & 1], d.stream));
    run.cur ^= 1;
    CU_CHECK(cudaGetLastError());
    return RT_OK;
}

// The rounds of every device, interleaved so that no device waits for another.  The host never waits for the round it
// has just enqueued: before round r + 2 it waits for round r's active count (one round of lookahead) and stops a device
// whose count was 0, so at most one empty round is launched and the GPU does not idle on the host.
int enqueue_render_adaptive(rt_gpu_ctx *ctx, std::vector<AdaptiveRun> &runs, const rt_render_params &rp, const rt_adaptive_params &ap,
                            const ViewSet *views, uint64_t &launches) {
    const uint32_t first = std::min(ap.min_samples, rp.samples);
    for (uint32_t round = 0;; ++round) {
        bool any = false;
        for (AdaptiveRun &run : runs) {
            if (run.finished) continue;
            if (run.done >= rp.samples) {
                run.finished = true;
                continue;
            }
            DeviceState &d = *run.d;
            if (round >= 2) {
                CU_CHECK(cudaSetDevice(d.device));
                CU_CHECK(cudaEventSynchronize(d.ev_round[round & 1]));  // round - 2's survivors
                if (d.h_active[round & 1] == 0) {
                    run.finished = true;
                    continue;
                }
            }
            const uint32_t k = round == 0 ? first : std::min(ap.step_samples, rp.samples - run.done);
            if (int rc = enqueue_adaptive_round(ctx, run, rp, ap, round, k, views, launches)) return rc;
            any = true;
        }
        if (!any) break;
    }
    for (AdaptiveRun &run : runs) {
        DeviceState &d = *run.d;
        CU_CHECK(cudaSetDevice(d.device));
        CU_CHECK(cudaEventRecord(d.ev_end, d.stream));
        CU_CHECK(cudaMemcpyAsync(d.h_stats, d.stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream));
    }
    return RT_OK;
}

}  // namespace

extern "C" {

const char *rt_gpu_last_error(void) { return g_last_error.c_str(); }
int rt_gpu_abi_version(void) { return RT_GPU_ABI_VERSION; }

int rt_gpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

namespace {
int create_devices(rt_gpu_ctx *ctx, int n_gpus, int first_device) {
    for (int i = 0; i < n_gpus; ++i) {
        ctx->devs.emplace_back(new DeviceState());
        DeviceState *d = ctx->devs.back().get();
        d->device = first_device + i;
        CU_CHECK(cudaSetDevice(d->device));
        cudaDeviceProp prop;
        CU_CHECK(cudaGetDeviceProperties(&prop, d->device));
        if (prop.major < 10)
            return fail(RT_ERR_NO_DEVICE, std::string("rt_gpu_create: device '") + prop.name +
                                              "' is not sm_100+ (kernels are built for sm_100a only)");
        d->sm_count = prop.multiProcessorCount;
        CU_CHECK(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
        CU_CHECK(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
        CU_CHECK(cudaStreamCreateWithFlags(&d->stream2, cudaStreamNonBlocking));
        CU_CHECK(cudaEventCreateWithFlags(&d->ev_a, cudaEventDisableTiming));
        CU_CHECK(cudaEventCreateWithFlags(&d->ev_b, cudaEventDisableTiming));
        CU_CHECK(cudaEventCreateWithFlags(&d->ev_light, cudaEventDisableTiming));
        CU_CHECK(cudaEventCreateWithFlags(&d->ev_copied, cudaEventDisableTiming));
        CU_CHECK(cudaEventCreate(&d->ev_begin));
        CU_CHECK(cudaEventCreate(&d->ev_end));
        CU_CHECK(cudaEventCreate(&d->ev_red0));
        CU_CHECK(cudaEventCreate(&d->ev_red1));
        CU_CHECK(cudaMallocHost(reinterpret_cast<void **>(&d->h_stats), 4 * sizeof(unsigned long long)));
        std::memset(d->h_stats, 0, 4 * sizeof(unsigned long long));
        CU_CHECK(cudaMallocHost(reinterpret_cast<void **>(&d->h_counters), sizeof(rtb::Counters)));
        CU_CHECK(cudaMallocHost(reinterpret_cast<void **>(&d->h_active), 2 * sizeof(uint32_t)));
        for (cudaEvent_t &e : d->ev_round) CU_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        int occ_e = 0, occ_s = 0;
        // experiment knob: shared-memory carve-out of k_extend in percent of the maximum (the rest of the 256 KB is L1)
        if (const char *e = std::getenv("RT_EXT_CARVEOUT"))
            CU_CHECK(cudaFuncSetAttribute(RT_K_EXTEND, cudaFuncAttributePreferredSharedMemoryCarveout, std::atoi(e)));
        CU_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_e, RT_K_EXTEND, rt::kExtendThreads, 0));
        CU_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_s, rt::k_shade, rt::kShadeThreads, 0));
        // experiment knobs: resident CTAs per SM of the two persistent kernels (default: all that fit)
        if (const char *e = std::getenv("RT_EXT_CTAS_PER_SM")) occ_e = std::min(occ_e, std::max(1, std::atoi(e)));
        if (const char *e = std::getenv("RT_SHADE_CTAS_PER_SM")) occ_s = std::min(occ_s, std::max(1, std::atoi(e)));
        int occ_l = 0;
        CU_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_l, rt::k_lightpdf_list, rt::kLightThreads, 0));
        d->light_blocks = d->sm_count * std::max(occ_l, 1);
        d->extend_blocks = d->sm_count * std::max(occ_e, 1);
        d->shade_blocks = d->sm_count * std::max(occ_s, 1);
    }
    if (n_gpus > 1) {
        if (!g_nccl.load()) return fail(RT_ERR_NCCL, "rt_gpu_create: libnccl.so.2 could not be loaded for a multi-device handle");
        std::vector<int> ids;
        for (auto &d : ctx->devs) ids.push_back(d->device);
        ctx->comms.assign(n_gpus, nullptr);
        const int rc = g_nccl.CommInitAll(ctx->comms.data(), n_gpus, ids.data());
        if (rc != 0) {
            ctx->comms.clear();
            return fail(RT_ERR_NCCL, std::string("ncclCommInitAll: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
        }
    }
    return RT_OK;
}
}  // namespace

int rt_gpu_create(rt_gpu_ctx **out, int n_gpus, int first_device) {
    if (!out || n_gpus < 1 || first_device < 0) return fail(RT_ERR_INVALID_ARG, "rt_gpu_create: bad arguments");
    *out = nullptr;
    const int have = rt_gpu_device_count();
    if (have < first_device + n_gpus)
        return fail(RT_ERR_NO_DEVICE, "rt_gpu_create: " + std::to_string(first_device + n_gpus) +
                                          " CUDA device(s) required, " + std::to_string(have) +
                                          " usable (this backend has no CPU path)");
    rt_gpu_ctx *ctx = new rt_gpu_ctx();
    if (int rc = create_devices(ctx, n_gpus, first_device)) {
        const std::string why = g_last_error;
        rt_gpu_destroy(ctx);  // streams, events, pinned memory and communicators built so far
        g_last_error = why;
        return rc;
    }
    *out = ctx;
    return RT_OK;
}

void rt_gpu_destroy(rt_gpu_ctx *ctx) {
    if (!ctx) return;
    // also the cleanup of a partially constructed handle (rt_gpu_create's error paths): every member may be null
    for (auto &dp : ctx->devs) {  // the device work (incl. a reduce in flight) ends before the communicators go
        if (!dp || !dp->stream) continue;
        cudaSetDevice(dp->device);
        cudaStreamSynchronize(dp->stream);
        if (dp->stream2) cudaStreamSynchronize(dp->stream2);
    }
    for (ncclComm_t c : ctx->comms)
        if (c) g_nccl.CommDestroy(c);
    for (auto &dp : ctx->devs) {
        if (!dp) continue;
        DeviceState &d = *dp;
        cudaSetDevice(d.device);
        d.qnodes4.release(); d.lqnodes4.release(); d.q4split.release(); d.qnodes8.release(); d.lqnodes8.release(); d.tprims.release(); d.tlights.release(); d.temit.release(); d.tris.release(); d.ltris.release(); d.lsample.release(); d.attrs.release();
        d.tangents.release(); d.light_extra.release(); d.materials.release(); d.textures.release();
        d.texels.release(); d.lut.release();
        d.arena.release(); d.means.release(); d.accum.release();
        if (d.h_stats) cudaFreeHost(d.h_stats);
        if (d.h_means) cudaFreeHost(d.h_means);
        if (d.h_stage) cudaFreeHost(d.h_stage);
        if (d.h_counters) cudaFreeHost(d.h_counters);
        if (d.h_active) cudaFreeHost(d.h_active);
        d.alist.release(); d.awords.release(); d.acounts.release(); d.actr.release(); d.aerr.release();
        d.in_pos.release(); d.in_nrm.release(); d.in_uv.release(); d.in_tan.release(); d.in_mat.release(); d.build_scratch.release(); d.refit_scratch.release();
        d.counters.release(); d.stats.release();
        d.prim_ids.release(); d.rgb8.release(); d.cams.release();
        d.aov_slots.release(); d.aov_sums.release(); d.aov_means.release();
        for (cudaEvent_t e : d.event_pool) cudaEventDestroy(e);
        for (cudaEvent_t e : {d.ev_begin, d.ev_end, d.ev_red0, d.ev_red1, d.ev_a, d.ev_b, d.ev_light, d.ev_round[0], d.ev_round[1]})
            if (e) cudaEventDestroy(e);
        if (d.stream2) cudaStreamDestroy(d.stream2);
        if (d.ev_copied) cudaEventDestroy(d.ev_copied);
        if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    cudaGetLastError();
    delete ctx;
}

int rt_gpu_upload_scene(rt_gpu_ctx *ctx, const rt_scene_desc *scene) {
    if (!ctx || !scene) return fail(RT_ERR_INVALID_ARG, "rt_gpu_upload_scene: null argument");
    if (scene->abi_version != RT_GPU_ABI_VERSION) return fail(RT_ERR_INVALID_ARG, "rt_gpu_upload_scene: ABI version mismatch");
    // structural validation (ids in range, arrays present) before anything is dereferenced
    if (scene->n_tris > 0 && (!scene->tri_pos || !scene->tri_normals || !scene->tri_uv || !scene->tri_material))
        return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: null per-triangle array with n_tris > 0");
    if ((scene->n_materials > 0 && !scene->materials) || (scene->n_textures > 0 && !scene->textures) ||
        (scene->texel_bytes > 0 && !scene->texels))
        return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: null material / texture array");
    if (scene->env_texture > scene->n_textures) return fail(RT_ERR_BAD_SCENE, "environment texture id out of range");
    for (const rt_bvh_desc *b : {&scene->scene_bvh, &scene->light_bvh})
        if ((b->n_nodes > 0 && !b->nodes) || (b->n_objects > 0 && !b->objects))
            return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: null BVH array");
    for (uint32_t i = 0; i < scene->n_tris; ++i)
        if (scene->tri_material[i] >= scene->n_materials) return fail(RT_ERR_BAD_SCENE, "material id out of range");
    for (const rt_bvh_desc *b : {&scene->scene_bvh, &scene->light_bvh})
        if (const char *why = bvh_problem(*b, scene->n_tris)) return fail(RT_ERR_BAD_SCENE, why);
    for (uint32_t i = 0; i < scene->n_materials; ++i) {
        const rt_material &m = scene->materials[i];
        for (int32_t t : {m.color_tex, m.emissive_tex, m.metallic_roughness_tex, m.normal_tex})
            if (t < -1 || t >= static_cast<int32_t>(scene->n_textures)) return fail(RT_ERR_BAD_SCENE, "texture id out of range");
    }
    for (uint32_t i = 0; i < scene->n_textures; ++i) {
        const rt_texture &t = scene->textures[i];
        if (!t.width || !t.height || t.offset + static_cast<uint64_t>(t.width) * t.height * 4 > scene->texel_bytes)
            return fail(RT_ERR_BAD_SCENE, "texture extent out of range");
    }
    rt::PackedScene &packed = ctx->packed;
    const char *keep_env = std::getenv("RT_KEEP_HOST_BVH");  // A/B switch for measurements
    const bool keep = (scene->flags & RT_SCENE_KEEP_HOST_BVH) || (keep_env && std::atoi(keep_env) != 0);
    if ((scene->flags & RT_SCENE_KEEP_HOST_BVH) && scene->scene_bvh.n_nodes == 0 && scene->n_tris > 0)
        return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_scene: RT_SCENE_KEEP_HOST_BVH without a scene BVH");
    const auto t_pack0 = std::chrono::steady_clock::now();
    double phase[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    rt::pack_times() = std::getenv("RT_TIMING") ? phase : nullptr;
    struct ResetTimes {
        ~ResetTimes() { rt::pack_times() = nullptr; }
    } reset_times;
    // Default: the scene BVH, triangles and attributes are built on the device (gpu_build.cuh); the host packs only the
    // light BVH, the materials and the textures.  The host builder (sah_build.h) remains for RT_SCENE_KEEP_HOST_BVH, for
    // the 8-wide build and as the A/B reference (RT_HOST_BUILD=1).
    const char *host_env = std::getenv("RT_HOST_BUILD");
    const bool device_build = !keep && !RT_EXT_WIDE8 && !(host_env && std::atoi(host_env) != 0);
    if (int rc = rt::pack_scene(*scene, packed, !keep, RT_EXT_WIDE8 ? rt::RT_PACK_Q8 : rt::RT_PACK_Q4, !device_build)) return fail(rc, "rt_gpu_upload_scene: scene cannot be re-packed (inner node with objects, depth > 64, non-finite box, or a 4-wide tree whose traversal needs more than RT_EXT_STACK_CAP stack entries)");
    const auto t_pack1 = std::chrono::steady_clock::now();
    double t_h2d = 0.0, t_build = 0.0;
    for (auto &d : ctx->devs) {
        if (device_build) {
            const auto tb0 = std::chrono::steady_clock::now();
            if (int rc = device_build_scene(*d, *scene, &t_h2d)) return rc;
            t_build = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb0).count();
        }
        if (int rc = upload_to_device(*d, *scene, packed, device_build)) return rc;
    }
    if (std::getenv("RT_TIMING")) {
        const auto t_up = std::chrono::steady_clock::now();
        if (device_build)
            std::fprintf(stderr, "rt_gpu_upload_scene: device build %.2f ms (of which H2D of the host arrays %.2f ms): %u levels, depth %u, %u wide nodes, stack need %u\n",
                         t_build, t_h2d, ctx->devs[0]->built_info[7], ctx->devs[0]->built_info[5], ctx->devs[0]->built_info[2], ctx->devs[0]->built_info[4]);
        std::fprintf(stderr,
                     "rt_gpu_upload_scene: re-pack %.1f ms (SAH build %.1f, triangles + binary nodes %.1f, collapse %.1f, quantise %.1f, "
                     "attributes %.1f, materials/texels %.1f; the light BVHs are inside the middle three), H2D %.1f ms\n",
                     std::chrono::duration<double, std::milli>(t_pack1 - t_pack0).count(), phase[0], phase[1], phase[2], phase[3], phase[5],
                     phase[6], std::chrono::duration<double, std::milli>(t_up - t_pack1).count());
    }
    ctx->ray_depth = scene->ray_depth;
    ctx->have_scene = true;
    ctx->have_render = false;
    ctx->adaptive = ctx->adaptive_sums = false;
    ctx->text_scene = false;
    return RT_OK;
}

int rt_gpu_update_geometry(rt_gpu_ctx *ctx, const rt_geometry_update *u) {
    if (!ctx || !u) return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: null argument");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_gpu_update_geometry: no scene uploaded");
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: a text scene has no triangle geometry to update");
    const DeviceState &d0 = *ctx->devs[0];
    if (d0.built_info[6] != 1)
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: the scene BVH was not built on the device (RT_SCENE_KEEP_HOST_BVH, "
                                        "RT_KEEP_HOST_BVH, RT_HOST_BUILD or the 8-wide library): re-upload the scene instead");
    if (u->n_tris != d0.built_info[0]) return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: n_tris differs from the uploaded scene's");
    if (u->n_tris > 0 && (!u->tri_pos || !u->tri_normals))
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: null tri_pos / tri_normals with n_tris > 0");
    const rt_bvh_desc &lb = u->light_bvh;
    if ((lb.n_nodes > 0 && !lb.nodes) || (lb.n_objects > 0 && !lb.objects)) return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: null BVH array");
    if (lb.n_objects != d0.scene.n_lights)
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: the light BVH has another number of objects than the uploaded one");
    if (const char *why = bvh_problem(lb, u->n_tris)) return fail(RT_ERR_INVALID_ARG, std::string("rt_gpu_update_geometry: ") + why);
    // the light side, as rt_gpu_upload_scene packs it for a device-built scene (rt::pack_scene with !keep)
    rt_scene_desc sc{};
    sc.abi_version = RT_GPU_ABI_VERSION;
    sc.n_tris = u->n_tris;
    sc.tri_pos = u->tri_pos;
    sc.light_bvh = lb;
    rt::PackedScene &packed = ctx->packed;
    if (rt::pack_lights(sc, packed, true, rt::RT_PACK_Q4))
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_update_geometry: the light BVH cannot be re-packed (inner node with objects, depth > 64, "
                                        "or a traversal that needs more than RT_EXT_STACK_CAP stack entries)");
    // from here on the device arrays change: a failure leaves no scene
    for (auto &dp : ctx->devs) {
        DeviceState &d = *dp;
        std::string phases;
        const auto t0 = std::chrono::steady_clock::now();
        int rc = device_refit_scene(d, *u, phases);
        if (rc == RT_OK) rc = upload_lights(d, packed, lb.n_objects);
        if (rc == RT_OK) rc = split_nodes(d, d.built_info[2], packed.light.qnodes4.size());
        if (rc == RT_OK) {
            const cudaError_t e = cudaStreamSynchronize(d.stream);
            if (e != cudaSuccess) rc = fail(RT_ERR_CUDA, std::string("rt_gpu_update_geometry: ") + cudaGetErrorString(e));
        }
        if (rc != RT_OK) {
            ctx->have_scene = false;
            return rc;
        }
        if (std::getenv("RT_TIMING"))
            std::fprintf(stderr, "rt_gpu_update_geometry: device %d %.3f ms (phases, serialised:%s)\n", d.device,
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), phases.c_str());
    }
    return RT_OK;
}

int rt_gpu_upload_text_scene(rt_gpu_ctx *ctx, const rt_text_scene *scene) {
    if (!ctx || !scene) return fail(RT_ERR_INVALID_ARG, "rt_gpu_upload_text_scene: null argument");
    if (scene->abi_version != RT_GPU_ABI_VERSION) return fail(RT_ERR_INVALID_ARG, "rt_gpu_upload_text_scene: ABI version mismatch");
    if (scene->n_prims > RT_TEXT_MAX_PRIMS || scene->n_lights > RT_TEXT_MAX_LIGHTS || scene->ray_depth > RT_TEXT_MAX_DEPTH ||
        scene->shading > RT_SHADE_PATH || (scene->n_prims && !scene->prims) || (scene->n_lights && !scene->lights))
        return fail(RT_ERR_BAD_SCENE, "rt_gpu_upload_text_scene: too many primitives / lights, depth > 16 or unknown shading");
    std::vector<rt_text_prim> prims(scene->prims, scene->prims + scene->n_prims);
    std::vector<rt_text_light> lights(scene->lights, scene->lights + scene->n_lights);
    std::vector<uint32_t> emitters;
    for (uint32_t i = 0; i < scene->n_prims; ++i) {
        const rt_text_prim &p = prims[i];
        if (p.kind > RT_PRIM_TRIANGLE || p.material > RT_MAT_DIELECTRIC) return fail(RT_ERR_BAD_SCENE, "unknown primitive kind / material");
        const bool emits = p.emission[0] != 0.0f || p.emission[1] != 0.0f || p.emission[2] != 0.0f;
        if (emits && p.kind != RT_PRIM_PLANE) emitters.push_back(i);  // an unbounded plane cannot be area-sampled
    }
    for (auto &dp : ctx->devs) {
        DeviceState &d = *dp;
        CU_CHECK(cudaSetDevice(d.device));
        if (int rc = d.tprims.upload(prims, d.stream)) return rc;
        if (int rc = d.tlights.upload(lights, d.stream)) return rc;
        if (int rc = d.temit.upload(emitters, d.stream)) return rc;
        rtt::TextScene &t = d.tscene;
        t.prims = d.tprims.p;
        t.lights = d.tlights.p;
        t.emitters = d.temit.p;
        t.n_prims = scene->n_prims;
        t.n_lights = scene->n_lights;
        t.n_emitters = static_cast<uint32_t>(emitters.size());
        t.ray_depth = scene->ray_depth;
        t.shading = scene->shading;
        for (int k = 0; k < 3; ++k) {
            t.bg[k] = scene->bg_color[k];
            t.ambient[k] = scene->ambient[k];
        }
        t.eps = scene->eps;
        d.tcamera = scene->camera;
        CU_CHECK(cudaStreamSynchronize(d.stream));
    }
    ctx->ray_depth = scene->ray_depth;
    ctx->have_scene = true;
    ctx->have_render = false;
    ctx->adaptive = ctx->adaptive_sums = false;
    ctx->text_scene = true;
    return RT_OK;
}

namespace {

// The per-pixel sums of every device reduced (sum) to device 0 in one NCCL group; with_counts adds the adaptive
// render's per-pixel sample counts (each device's are 0 outside its pixel range).
int reduce_to_device0(rt_gpu_ctx *ctx, size_t n_pix, bool with_counts) {
    const int n = static_cast<int>(ctx->devs.size());
    for (auto &d : ctx->devs) {
        CU_CHECK(cudaSetDevice(d->device));
        CU_CHECK(cudaEventRecord(d->ev_red0, d->stream));
    }
    g_nccl.GroupStart();
    for (int g = 0; g < n; ++g) {
        DeviceState &d = *ctx->devs[g];
        int rc = g_nccl.Reduce(d.accum.p, d.accum.p, n_pix * 4, kNcclFloat32, kNcclSum, 0, ctx->comms[g], d.stream);
        if (rc == 0 && with_counts) rc = g_nccl.Reduce(d.acounts.p, d.acounts.p, n_pix, kNcclUint32, kNcclSum, 0, ctx->comms[g], d.stream);
        if (rc != 0) {
            g_nccl.GroupEnd();
            return fail(RT_ERR_NCCL, std::string("ncclReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
        }
    }
    if (int rc = g_nccl.GroupEnd()) return fail(RT_ERR_NCCL, std::string("ncclGroupEnd: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"));
    for (auto &d : ctx->devs) {
        CU_CHECK(cudaSetDevice(d->device));
        CU_CHECK(cudaEventRecord(d->ev_red1, d->stream));
    }
    return RT_OK;
}

// Waits for every device, gathers the work counters and timings of the render into ctx->stats.
int finish_render(rt_gpu_ctx *ctx, const rt_render_params &rp, uint64_t launches) {
    const int n = static_cast<int>(ctx->devs.size());
    rt_stats st;
    std::memset(&st, 0, sizeof st);
    for (int g = 0; g < n; ++g) {
        DeviceState &d = *ctx->devs[g];
        if (rp.mode == RT_MODE_PRIMARY_IDS && g > 0) continue;
        CU_CHECK(cudaSetDevice(d.device));
        CU_CHECK(cudaStreamSynchronize(d.stream));
        float ms = 0.0f;
        CU_CHECK(cudaEventElapsedTime(&ms, d.ev_begin, d.ev_end));
        st.render_ms = std::max(st.render_ms, static_cast<double>(ms));
        if (n > 1 && rp.mode == RT_MODE_BEAUTY) {
            CU_CHECK(cudaEventElapsedTime(&ms, d.ev_red0, d.ev_red1));
            st.reduce_ms = std::max(st.reduce_ms, static_cast<double>(ms));
        }
        const unsigned long long *hs = d.h_stats;
        st.extension_rays += hs[0];
        st.light_pdf_rays += hs[1];
        st.shades += hs[2];
        st.samples += hs[3];
        if (ctx->profiling && std::getenv("RT_TIMING") && d.counters.p) {  // queue and light-list sizes of the last batch
            std::vector<uint32_t> hc(d.counters.n);
            cudaMemcpy(hc.data(), d.counters.p, d.counters.n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
            const uint32_t qd = std::max(d.scene.ray_depth, 1u);
            std::string line = "rt_gpu queue sizes (last batch), bounce: rays / listed for k_lightpdf:";
            for (uint32_t b = 0; b <= qd && (3 * qd + 1 + b) * rt::kCounterStride < hc.size(); ++b)
                line += " " + std::to_string(hc[b * rt::kCounterStride]) + "/" + std::to_string(hc[(3 * qd + 1 + b) * rt::kCounterStride]);
            std::fprintf(stderr, "%s\n", line.c_str());
        }
        if (ctx->profiling) {
            double per_kind[K_COUNT] = {0};
            for (size_t i = 1; i < d.marks.size(); ++i) {
                float dt = 0.0f;
                cudaEventElapsedTime(&dt, d.marks[i - 1].first, d.marks[i].first);
                if (d.marks[i].second >= 0) per_kind[d.marks[i].second] += dt;
            }
            for (int k = 0; k < K_COUNT; ++k) st.kernel_ms[k] = std::max(st.kernel_ms[k], per_kind[k]);
        }
    }
    st.kernel_launches = launches;
    ctx->stats = st;
    return RT_OK;
}

// Pixels of the last render's image: width * height, times the views of a multi-view render
size_t last_pixels(const rt_gpu_ctx *ctx) {
    return static_cast<size_t>(ctx->last.width) * ctx->last.height * std::max(ctx->last_views, 1u);
}

// The render of rt_gpu_render (views == nullptr) and rt_gpu_render_views over every device of the handle; rp is
// validated and its sample_end / pixel_end resolved.
int render_on_devices(rt_gpu_ctx *ctx, const rt_render_params &rp, const ViewSet *views) {
    const int n = static_cast<int>(ctx->devs.size());
    const uint32_t total = rp.sample_end - rp.sample_begin;
    uint64_t launches = 0;
    // sample-split: device g renders [begin + g*total/n, begin + (g+1)*total/n) of every pixel.  With fewer samples
    // than devices the image is split instead: device g renders all samples of a contiguous range of the pixels
    // (the other pixels of its buffer stay 0, so the same reduce(sum) merges the tiles).
    const bool tile_split = n > 1 && total < static_cast<uint32_t>(n) && rp.mode == RT_MODE_BEAUTY;
    const uint64_t n_px = rp.pixel_end - rp.pixel_begin;
    for (int g = 0; g < n; ++g) {
        uint32_t sb = rp.sample_begin + static_cast<uint32_t>(static_cast<uint64_t>(total) * g / n);
        uint32_t se = rp.sample_begin + static_cast<uint32_t>(static_cast<uint64_t>(total) * (g + 1) / n);
        rt_render_params local = rp;
        if (tile_split) {
            sb = rp.sample_begin;
            se = rp.sample_end;
            local.pixel_begin = rp.pixel_begin + static_cast<uint32_t>(n_px * g / n);
            local.pixel_end = rp.pixel_begin + static_cast<uint32_t>(n_px * (g + 1) / n);
            if (local.pixel_end == local.pixel_begin) se = sb;  // nothing for this device: zero buffer only
        }
        if (rp.mode == RT_MODE_PRIMARY_IDS && g > 0) continue;  // ids: device 0 only
        DeviceState &dg = *ctx->devs[g];
        if (ctx->text_scene) {
            if (int rc = enqueue_text_render(ctx, dg, g, local, sb, se, launches)) return rc;
        } else if (int rc = enqueue_render(ctx, dg, g, local, sb, se, views, launches)) {
            return rc;
        }
        // the work counters travel on the stream into pinned memory: no second synchronising copy after the render
        CU_CHECK(cudaMemcpyAsync(dg.h_stats, dg.stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, dg.stream));
    }
    const size_t n_pix = static_cast<size_t>(rp.width) * rp.height * (views ? views->cams.size() : 1);
    if (n > 1 && rp.mode == RT_MODE_BEAUTY)
        if (int rc = reduce_to_device0(ctx, n_pix, false)) return rc;
    if (int rc = finish_render(ctx, rp, launches)) return rc;
    ctx->last = rp;
    ctx->last_views = views ? static_cast<uint32_t>(views->cams.size()) : 0u;
    ctx->have_render = true;
    ctx->adaptive = false;
    if (rp.mode == RT_MODE_BEAUTY) ctx->adaptive_sums = false;
    return RT_OK;
}

// The checks of the views of rt_gpu_render_views (and rt_gpu_render_views_adaptive): views, stacked image size, the
// 32-bit key and finite cameras.  Fills vs with the device cameras.
int check_views(const rt_render_params &rp, const rt_views &views, const std::string &who, ViewSet &vs) {
    if (views.n_views == 0 || !views.cameras) return fail(RT_ERR_INVALID_ARG, who + ": no views / null cameras");
    const uint64_t per_view = static_cast<uint64_t>(rp.width) * rp.height, V = views.n_views;
    if (per_view == 0 || per_view > 0x7FFFFFFFull || per_view * V > 0x7FFFFFFFull)
        return fail(RT_ERR_INVALID_ARG, who + ": illegal image size (the stacked image has n_views * width * height pixels)");
    if ((views.view_base + V) * per_view > (1ull << 32))
        return fail(RT_ERR_INVALID_ARG, who + ": (view_base + n_views) * width * height exceeds the 32-bit pixel key");
    for (uint32_t v = 0; v < views.n_views; ++v) {
        const rt_camera &c = views.cameras[v];
        bool finite = std::isfinite(c.fov_x);
        for (int k = 0; k < 3; ++k)
            finite = finite && std::isfinite(c.position[k]) && std::isfinite(c.right[k]) && std::isfinite(c.up[k]) && std::isfinite(c.forward[k]);
        if (!finite) return fail(RT_ERR_INVALID_ARG, who + ": camera " + std::to_string(v) + " has a non-finite value");
    }
    vs.view_base = views.view_base;
    vs.cams.clear();
    for (uint32_t v = 0; v < views.n_views; ++v) vs.cams.push_back(make_camera(views.cameras[v], rp.width, rp.height));
    return RT_OK;
}

// The checks of the projections of rt_gpu_render_projected (one per view of vs, already checked by check_views).
// Fills vs.projs.  Fields a kind does not use are not looked at.
int check_projections(const rt_projection *projections, const std::string &who, ViewSet &vs) {
    vs.projs.clear();
    for (size_t v = 0; v < vs.cams.size(); ++v) {
        const rt_projection &p = projections[v];
        const std::string at = who + ": projection " + std::to_string(v);
        rt::Projection q{p.kind, 0.0f, 0.0f, 0.0f, 0.0f};
        if (p.kind == RT_PROJ_THIN_LENS) {
            if (!std::isfinite(p.aperture_radius) || !std::isfinite(p.focus_distance)) return fail(RT_ERR_INVALID_ARG, at + " has a non-finite value");
            if (p.aperture_radius < 0.0f) return fail(RT_ERR_INVALID_ARG, at + ": aperture_radius < 0");
            if (p.aperture_radius > 0.0f && !(p.focus_distance > 0.0f))
                return fail(RT_ERR_INVALID_ARG, at + ": focus_distance <= 0 with a non-zero aperture");
            q.aperture_radius = p.aperture_radius;
            q.focus_distance = p.focus_distance;
        } else if (p.kind == RT_PROJ_ORTHOGRAPHIC) {
            if (!std::isfinite(p.half_width) || !std::isfinite(p.half_height)) return fail(RT_ERR_INVALID_ARG, at + " has a non-finite value");
            if (!(p.half_width > 0.0f) || !(p.half_height > 0.0f)) return fail(RT_ERR_INVALID_ARG, at + ": half_width / half_height <= 0");
            q.half_width = p.half_width;
            q.half_height = p.half_height;
        } else if (p.kind != RT_PROJ_PINHOLE && p.kind != RT_PROJ_EQUIRECT) {
            return fail(RT_ERR_INVALID_ARG, at + ": unknown kind " + std::to_string(p.kind));
        }
        vs.projs.push_back(q);
    }
    return RT_OK;
}

// The checks of an adaptive render's parameters over an image of n_pixels; resolves rp.pixel_end
int check_adaptive(rt_render_params &rp, const rt_adaptive_params &ap, uint64_t n_pixels, const std::string &who) {
    if (rp.mode != RT_MODE_BEAUTY) return fail(RT_ERR_INVALID_ARG, who + ": beauty renders only");
    if (rp.samples < 2) return fail(RT_ERR_INVALID_ARG, who + ": samples (the maximum spp) < 2");
    if (rp.sample_begin != 0 || rp.sample_end != 0)
        return fail(RT_ERR_INVALID_ARG, who + ": every pixel starts at sample 0 (sample_begin / sample_end must be 0)");
    if (rp.flags & RT_FLAG_ACCUMULATE) return fail(RT_ERR_INVALID_ARG, who + ": RT_FLAG_ACCUMULATE is not supported");
    if (ap.min_samples < 2 || ap.step_samples == 0 || !(ap.abs_floor > 0.0f) || !(ap.rel_error >= 0.0f))
        return fail(RT_ERR_INVALID_ARG, who + ": needs min_samples >= 2, step_samples >= 1, abs_floor > 0, rel_error >= 0");
    if (rp.pixel_end == 0) rp.pixel_end = static_cast<uint32_t>(n_pixels);
    if (rp.pixel_begin > rp.pixel_end || rp.pixel_end > n_pixels) return fail(RT_ERR_INVALID_ARG, who + ": illegal pixel range");
    return RT_OK;
}

// The adaptive render of rt_gpu_render_adaptive (views == nullptr) and rt_gpu_render_views_adaptive over every device of
// the handle; rp and ap are validated and rp.pixel_end resolved.
int render_adaptive_on_devices(rt_gpu_ctx *ctx, const rt_render_params &rp, const rt_adaptive_params &ap, const ViewSet *views) {
    const uint32_t n_views = views ? static_cast<uint32_t>(views->cams.size()) : 1u;
    const uint64_t n_pixels = static_cast<uint64_t>(rp.width) * rp.height * n_views;
    // every device adapts a contiguous part of the range (a pixel's decisions depend on its own sums only)
    const int n = static_cast<int>(ctx->devs.size());
    const uint64_t n_px = rp.pixel_end - rp.pixel_begin;
    std::vector<AdaptiveRun> runs(n);
    ctx->have_render = false;  // the sums are being replaced
    for (int g = 0; g < n; ++g) {
        runs[g].d = ctx->devs[g].get();
        const size_t b = rp.pixel_begin + n_px * g / n, e = rp.pixel_begin + n_px * (g + 1) / n;
        if (int rc = setup_adaptive(ctx, runs[g], rp, b, e, views)) return rc;
    }
    uint64_t launches = 0;
    if (int rc = enqueue_render_adaptive(ctx, runs, rp, ap, views, launches)) return rc;
    if (n > 1)
        if (int rc = reduce_to_device0(ctx, static_cast<size_t>(n_pixels), true)) return rc;
    if (int rc = finish_render(ctx, rp, launches)) return rc;
    if (std::getenv("RT_TIMING")) {  // contiguous tiles are not load-balanced: the per-device times show by how much
        for (int g = 0; g < n; ++g) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, runs[g].d->ev_begin, runs[g].d->ev_end);
            std::fprintf(stderr, "rt_gpu adaptive: device %d pixels [%zu, %zu) %.2f ms, %llu samples\n", runs[g].d->device, runs[g].pix0,
                         runs[g].pix0 + runs[g].n_render, ms, static_cast<unsigned long long>(runs[g].d->h_stats[3]));
        }
    }
    ctx->last = rp;
    ctx->last_views = views ? n_views : 0u;
    ctx->last_adaptive = ap;
    ctx->have_render = true;
    ctx->adaptive = ctx->adaptive_sums = true;
    return RT_OK;
}

// rt_gpu_render_views (projections == nullptr) and the fixed form of rt_gpu_render_projected after their null checks
int render_views_checked(rt_gpu_ctx *ctx, const rt_render_params &params, const rt_views &views, const rt_projection *projections,
                         const std::string &who) {
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, who + ": no scene uploaded");
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, who + ": not available for course text scenes");
    rt_render_params rp = params;
    ViewSet vs;
    if (int rc = check_views(rp, views, who, vs)) return rc;
    if (projections)
        if (int rc = check_projections(projections, who, vs)) return rc;
    const uint64_t per_view = static_cast<uint64_t>(rp.width) * rp.height, V = views.n_views;
    if (rp.mode == RT_MODE_BEAUTY && rp.samples == 0) return fail(RT_ERR_INVALID_ARG, who + ": samples == 0");
    if (rp.sample_end == 0) rp.sample_end = rp.samples;
    if (rp.sample_begin > rp.sample_end) return fail(RT_ERR_INVALID_ARG, who + ": sample_begin > sample_end");
    const uint64_t n_pixels = per_view * V;
    if (rp.pixel_end == 0) rp.pixel_end = static_cast<uint32_t>(n_pixels);
    if (rp.pixel_begin > rp.pixel_end || rp.pixel_end > n_pixels) return fail(RT_ERR_INVALID_ARG, who + ": illegal pixel range");
    if ((rp.flags & RT_FLAG_ACCUMULATE) && rp.mode == RT_MODE_BEAUTY &&
        (!ctx->have_render || ctx->adaptive_sums || ctx->last.width != rp.width || ctx->last.height != rp.height ||
         std::max(ctx->last_views, 1u) != views.n_views))
        return fail(RT_ERR_INVALID_ARG, who + ": RT_FLAG_ACCUMULATE needs a previous render of the same width, height and n_views");
    return render_on_devices(ctx, rp, &vs);
}

// rt_gpu_render_views_adaptive (projections == nullptr) and the adaptive form of rt_gpu_render_projected after their
// null checks
int render_views_adaptive_checked(rt_gpu_ctx *ctx, const rt_render_params &params, const rt_views &views, const rt_projection *projections,
                                  const rt_adaptive_params &ap, const std::string &who) {
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, who + ": no scene uploaded");
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, who + ": not available for course text scenes");
    rt_render_params rp = params;
    ViewSet vs;
    if (int rc = check_views(rp, views, who, vs)) return rc;
    if (projections)
        if (int rc = check_projections(projections, who, vs)) return rc;
    if (int rc = check_adaptive(rp, ap, static_cast<uint64_t>(rp.width) * rp.height * views.n_views, who)) return rc;
    return render_adaptive_on_devices(ctx, rp, ap, &vs);
}

}  // namespace

int rt_gpu_render(rt_gpu_ctx *ctx, const rt_render_params *params) {
    if (!ctx || !params) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: null argument");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_gpu_render: no scene uploaded");
    rt_render_params rp = *params;
    if (rp.width == 0 || rp.height == 0 || static_cast<uint64_t>(rp.width) * rp.height > 0x7FFFFFFFull)
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: illegal image size");
    if (rp.mode == RT_MODE_BEAUTY && rp.samples == 0) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: samples == 0");
    if (rp.sample_end == 0) rp.sample_end = rp.samples;
    if (rp.sample_begin > rp.sample_end) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: sample_begin > sample_end");
    const uint64_t n_pixels = static_cast<uint64_t>(rp.width) * rp.height;
    if (rp.pixel_end == 0) rp.pixel_end = static_cast<uint32_t>(n_pixels);
    if (rp.pixel_begin > rp.pixel_end || rp.pixel_end > n_pixels) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: illegal pixel range");
    if ((rp.flags & RT_FLAG_ACCUMULATE) && rp.mode == RT_MODE_BEAUTY && ctx->adaptive_sums)
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: RT_FLAG_ACCUMULATE onto the sums of an adaptive render (per-pixel sample counts)");
    if ((rp.flags & RT_FLAG_ACCUMULATE) && rp.mode == RT_MODE_BEAUTY && ctx->have_render && ctx->last_views != 0 &&
        (ctx->last_views != 1 || ctx->last.width != rp.width || ctx->last.height != rp.height))
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_render: RT_FLAG_ACCUMULATE onto the sums of a multi-view render of another shape");
    return render_on_devices(ctx, rp, nullptr);
}

int rt_gpu_render_views(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views) {
    if (!ctx || !params || !views) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render_views: null argument");
    return render_views_checked(ctx, *params, *views, nullptr, "rt_gpu_render_views");
}

int rt_gpu_render_adaptive(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_adaptive_params *ap) {
    if (!ctx || !params || !ap) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render_adaptive: null argument");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_gpu_render_adaptive: no scene uploaded");
    rt_render_params rp = *params;
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, "rt_gpu_render_adaptive: not available for course text scenes");
    if (rp.width == 0 || rp.height == 0 || static_cast<uint64_t>(rp.width) * rp.height > 0x7FFFFFFFull)
        return fail(RT_ERR_INVALID_ARG, "rt_gpu_render_adaptive: illegal image size");
    if (int rc = check_adaptive(rp, *ap, static_cast<uint64_t>(rp.width) * rp.height, "rt_gpu_render_adaptive")) return rc;
    return render_adaptive_on_devices(ctx, rp, *ap, nullptr);
}

int rt_gpu_render_views_adaptive(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views, const rt_adaptive_params *ap) {
    const std::string who = "rt_gpu_render_views_adaptive";
    if (!ctx || !params || !views || !ap) return fail(RT_ERR_INVALID_ARG, who + ": null argument");
    return render_views_adaptive_checked(ctx, *params, *views, nullptr, *ap, who);
}

int rt_gpu_render_projected(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views, const rt_projection *projections,
                            const rt_adaptive_params *ap) {
    const std::string who = "rt_gpu_render_projected";
    if (!ctx || !params || !views || !projections) return fail(RT_ERR_INVALID_ARG, who + ": null argument");
    if (!ap) return render_views_checked(ctx, *params, *views, projections, who);
    return render_views_adaptive_checked(ctx, *params, *views, projections, *ap, who);
}

int rt_gpu_render_aov(rt_gpu_ctx *ctx, const rt_render_params *params, const rt_views *views, const rt_projection *projections) {
    const std::string who = "rt_gpu_render_aov";
    if (!ctx || !params) return fail(RT_ERR_INVALID_ARG, who + ": null argument");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, who + ": no scene uploaded");
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, who + ": not available for course text scenes");
    if (projections && !views) return fail(RT_ERR_INVALID_ARG, who + ": projections need views");
    rt_render_params rp = *params;
    if (rp.mode != RT_MODE_BEAUTY && rp.mode != RT_MODE_PRIMARY_IDS) return fail(RT_ERR_INVALID_ARG, who + ": unknown mode");
    if (rp.sample_begin != 0 || rp.sample_end != 0)
        return fail(RT_ERR_INVALID_ARG, who + ": the samples are [0, samples) (sample_begin / sample_end must be 0)");
    if (rp.flags & RT_FLAG_ACCUMULATE) return fail(RT_ERR_INVALID_ARG, who + ": RT_FLAG_ACCUMULATE is not supported");
    ViewSet vs;
    if (views) {
        if (int rc = check_views(rp, *views, who, vs)) return rc;
        if (projections)
            if (int rc = check_projections(projections, who, vs)) return rc;
    } else if (rp.width == 0 || rp.height == 0 || static_cast<uint64_t>(rp.width) * rp.height > 0x7FFFFFFFull) {
        return fail(RT_ERR_INVALID_ARG, who + ": illegal image size");
    }
    if (rp.mode == RT_MODE_BEAUTY && rp.samples == 0) return fail(RT_ERR_INVALID_ARG, who + ": samples == 0");
    const uint64_t n_pixels = static_cast<uint64_t>(rp.width) * rp.height * (views ? views->n_views : 1u);
    if (rp.pixel_end == 0) rp.pixel_end = static_cast<uint32_t>(n_pixels);
    if (rp.pixel_begin > rp.pixel_end || rp.pixel_end > n_pixels) return fail(RT_ERR_INVALID_ARG, who + ": illegal pixel range");
    // device 0 only, as RT_MODE_PRIMARY_IDS: the sums are its own
    ctx->have_aov = false;
    DeviceState &d = *ctx->devs[0];
    uint64_t launches = 0;
    if (int rc = enqueue_render_aov(d, rp, views ? &vs : nullptr, launches)) return rc;
    CU_CHECK(cudaMemcpyAsync(d.h_stats, d.stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaStreamSynchronize(d.stream));
    rt_stats st;
    std::memset(&st, 0, sizeof st);
    float ms = 0.0f;
    CU_CHECK(cudaEventElapsedTime(&ms, d.ev_begin, d.ev_end));
    st.render_ms = ms;
    st.extension_rays = d.h_stats[0];
    st.samples = d.h_stats[3];
    st.kernel_launches = launches;
    ctx->aov_stats = st;
    ctx->aov_last = rp;
    ctx->aov_views = views ? views->n_views : 0u;
    ctx->aov_samples = rp.mode == RT_MODE_PRIMARY_IDS ? 1u : rp.samples;
    ctx->have_aov = true;
    return RT_OK;
}

int rt_gpu_readback_aov(rt_gpu_ctx *ctx, float *albedo, float *normal, float *emission, float *depth, float *coverage, rt_stats *stats) {
    const std::string who = "rt_gpu_readback_aov";
    if (!ctx) return fail(RT_ERR_INVALID_ARG, who + ": null handle");
    if (!ctx->have_aov) return fail(RT_ERR_NO_RENDER, who + ": no AOV render on this handle");
    DeviceState &d = *ctx->devs[0];
    CU_CHECK(cudaSetDevice(d.device));
    const size_t n = static_cast<size_t>(ctx->aov_last.width) * ctx->aov_last.height * std::max(ctx->aov_views, 1u);
    if (albedo || normal || emission || depth || coverage) {
        if (int rc = d.aov_means.alloc(11 * n)) return rc;
        const rt::AovPlanes sums{d.aov_sums.p, d.aov_sums.p + n, d.aov_sums.p + 2 * n};
        const uint32_t n32 = static_cast<uint32_t>(n);
        rt::k_aov_means<<<(n32 + 255) / 256, 256, 0, d.stream>>>(sums, static_cast<float>(ctx->aov_samples), n32, d.aov_means.p);
        CU_CHECK(cudaGetLastError());
        const float *m = d.aov_means.p;
        const struct {
            float *dst;
            const float *src;
            size_t count;
        } parts[5] = {{albedo, m, 3 * n}, {normal, m + 3 * n, 3 * n}, {emission, m + 6 * n, 3 * n}, {depth, m + 9 * n, n}, {coverage, m + 10 * n, n}};
        for (const auto &part : parts)
            if (part.dst) CU_CHECK(cudaMemcpyAsync(part.dst, part.src, part.count * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
        CU_CHECK(cudaStreamSynchronize(d.stream));
    }
    if (stats) *stats = ctx->aov_stats;
    return RT_OK;
}

int rt_gpu_readback_adaptive(rt_gpu_ctx *ctx, uint32_t *sample_counts, float *rel_error) {
    if (!ctx) return fail(RT_ERR_INVALID_ARG, "rt_gpu_readback_adaptive: null handle");
    if (!ctx->have_render || !ctx->adaptive) return fail(RT_ERR_NO_RENDER, "rt_gpu_readback_adaptive: the last render was not adaptive");
    const size_t n_pix = last_pixels(ctx);  // times the views after rt_gpu_render_views_adaptive
    if (sample_counts) {  // reduced to device 0
        DeviceState &d = *ctx->devs[0];
        CU_CHECK(cudaSetDevice(d.device));
        CU_CHECK(cudaMemcpy(sample_counts, d.acounts.p, n_pix * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    }
    if (rel_error) {  // gathered from every device's own range
        std::memset(rel_error, 0, n_pix * sizeof(float));
        for (auto &dp : ctx->devs) {
            DeviceState &d = *dp;
            if (d.apix1 <= d.apix0) continue;
            CU_CHECK(cudaSetDevice(d.device));
            CU_CHECK(cudaMemcpy(rel_error + d.apix0, d.aerr.p + d.apix0, (d.apix1 - d.apix0) * sizeof(float), cudaMemcpyDeviceToHost));
        }
    }
    return RT_OK;
}

int rt_gpu_readback(rt_gpu_ctx *ctx, float *rgb_mean, int32_t *prim_ids, rt_stats *stats) {
    if (!ctx) return fail(RT_ERR_INVALID_ARG, "rt_gpu_readback: null handle");
    if (!ctx->have_render) return fail(RT_ERR_NO_RENDER, "rt_gpu_readback: nothing rendered");
    DeviceState &d = *ctx->devs[0];
    CU_CHECK(cudaSetDevice(d.device));
    const size_t n_pix = last_pixels(ctx);
    if (rgb_mean) {
        if (ctx->last.mode != RT_MODE_BEAUTY) return fail(RT_ERR_NO_RENDER, "rt_gpu_readback: last render was not a beauty render");
        // the division and the float4 -> rgb packing run on the device (12 B per pixel cross the bus instead of 16);
        // the copy lands directly in the caller's buffer when that is pinned, else in chunks through a persistent
        // pinned staging buffer, each chunk's host memcpy overlapping the next chunk's DMA
        const size_t n_f = n_pix * 3;
        if (int rc = d.means.alloc(n_f)) return rc;
        const uint32_t np32 = static_cast<uint32_t>(n_pix);
        if (ctx->adaptive_sums)
            rt::k_means_counts<<<(np32 + 255) / 256, 256, 0, d.stream>>>(d.accum.p, d.acounts.p, np32, d.means.p);
        else
            rt::k_means<<<(np32 + 255) / 256, 256, 0, d.stream>>>(d.accum.p, static_cast<float>(ctx->last.samples), np32, d.means.p);
        CU_CHECK(cudaGetLastError());
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, rgb_mean) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned) {
            CU_CHECK(cudaMemcpyAsync(rgb_mean, d.means.p, n_f * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
            CU_CHECK(cudaStreamSynchronize(d.stream));
        } else {
            if (d.h_means_n < n_f) {
                if (d.h_means) cudaFreeHost(d.h_means);
                d.h_means = nullptr;
                d.h_means_n = 0;
                CU_CHECK(cudaMallocHost(reinterpret_cast<void **>(&d.h_means), n_f * sizeof(float)));
                d.h_means_n = n_f;
            }
            constexpr int kChunks = 4;
            size_t at[kChunks + 1];
            for (int c = 0; c <= kChunks; ++c) at[c] = n_f * c / kChunks;
            for (int c = 0; c < kChunks; ++c) {
                CU_CHECK(cudaMemcpyAsync(d.h_means + at[c], d.means.p + at[c], (at[c + 1] - at[c]) * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
                CU_CHECK(cudaEventRecord(c & 1 ? d.ev_red1 : d.ev_red0, d.stream));
                if (c > 0) {
                    CU_CHECK(cudaEventSynchronize((c - 1) & 1 ? d.ev_red1 : d.ev_red0));
                    std::memcpy(rgb_mean + at[c - 1], d.h_means + at[c - 1], (at[c] - at[c - 1]) * sizeof(float));
                }
            }
            CU_CHECK(cudaStreamSynchronize(d.stream));
            std::memcpy(rgb_mean + at[kChunks - 1], d.h_means + at[kChunks - 1], (at[kChunks] - at[kChunks - 1]) * sizeof(float));
        }
    }
    if (prim_ids) {
        if (ctx->last.mode != RT_MODE_PRIMARY_IDS) return fail(RT_ERR_NO_RENDER, "rt_gpu_readback: last render was not a primary-id render");
        CU_CHECK(cudaMemcpy(prim_ids, d.prim_ids.p, n_pix * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    if (stats) *stats = ctx->stats;
    return RT_OK;
}

int rt_gpu_accum_device_ptr(rt_gpu_ctx *ctx, void **dptr, size_t *n_floats) {
    if (!ctx || !dptr) return fail(RT_ERR_INVALID_ARG, "rt_gpu_accum_device_ptr: null argument");
    if (!ctx->have_render || ctx->last.mode != RT_MODE_BEAUTY) return fail(RT_ERR_NO_RENDER, "rt_gpu_accum_device_ptr: no beauty render");
    *dptr = ctx->devs[0]->accum.p;
    if (n_floats) *n_floats = last_pixels(ctx) * 4;
    return RT_OK;
}

int rt_gpu_readback_rgb8(rt_gpu_ctx *ctx, uint8_t *rgb8) {
    if (!ctx || !rgb8) return fail(RT_ERR_INVALID_ARG, "rt_gpu_readback_rgb8: null argument");
    if (!ctx->have_render || ctx->last.mode != RT_MODE_BEAUTY) return fail(RT_ERR_NO_RENDER, "rt_gpu_readback_rgb8: no beauty render");
    DeviceState &d = *ctx->devs[0];
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t n_pix = static_cast<uint32_t>(last_pixels(ctx));
    if (int rc = d.rgb8.alloc(static_cast<size_t>(n_pix) * 3)) return rc;
    if (ctx->adaptive_sums)
        rt::k_tonemap_counts<<<(n_pix + 255) / 256, 256, 0, d.stream>>>(d.accum.p, d.acounts.p, n_pix, d.rgb8.p);
    else
        rt::k_tonemap<<<(n_pix + 255) / 256, 256, 0, d.stream>>>(d.accum.p, static_cast<float>(ctx->last.samples), n_pix, d.rgb8.p);
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaMemcpyAsync(rgb8, d.rgb8.p, static_cast<size_t>(n_pix) * 3, cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaStreamSynchronize(d.stream));
    return RT_OK;
}

int rt_gpu_fp32_peak(rt_gpu_ctx *ctx, double *tflops) {
    if (!ctx || !tflops) return fail(RT_ERR_INVALID_ARG, "rt_gpu_fp32_peak: null argument");
    DeviceState &d = *ctx->devs[0];
    CU_CHECK(cudaSetDevice(d.device));
    if (int rc = d.lut.alloc(256)) return rc;
    const int iters = 1 << 14, threads = 256, blocks = d.sm_count * 8;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU_CHECK(cudaEventRecord(d.ev_red0, d.stream));
        rt::k_fma_peak<<<blocks, threads, 0, d.stream>>>(d.lut.p, 0.999f, 1e-4f, iters);
        CU_CHECK(cudaEventRecord(d.ev_red1, d.stream));
        CU_CHECK(cudaStreamSynchronize(d.stream));
        float ms = 0.0f;
        CU_CHECK(cudaEventElapsedTime(&ms, d.ev_red0, d.ev_red1));
        const double flops = 2.0 * 16.0 * iters * static_cast<double>(threads) * blocks;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) * 1e-12);
    }
    *tflops = best;
    return RT_OK;
}

int rt_gpu_debug_get_bvh(rt_gpu_ctx *ctx, int which, void *dst, size_t *bytes) {
    if (!ctx || !bytes) return fail(RT_ERR_INVALID_ARG, "rt_gpu_debug_get_bvh: null argument");
    if (!ctx->have_scene || ctx->text_scene) return fail(RT_ERR_NO_SCENE, "rt_gpu_debug_get_bvh: no triangle scene uploaded");
    DeviceState &d = *ctx->devs[0];
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t n = d.built_info[0], n_slots = d.built_info[1], n_wide = d.built_info[2];
    const bool dev = d.built_info[6] != 0;
    const void *src = nullptr;
    size_t sz = 0;
    switch (which) {
    case 0: src = d.built_info; sz = sizeof d.built_info; break;
    case 1: if (dev) { src = d.built.nodes; sz = static_cast<size_t>(n_slots) * sizeof(rt_bvh_node); } break;
    case 2: if (dev) { src = d.built.idx[d.built_parity]; sz = static_cast<size_t>(n) * 4; } break;
    case 3: if (dev) { src = d.qnodes4.p; sz = static_cast<size_t>(n_wide) * sizeof(QNode4); } break;
    case 4: if (dev) { src = d.tris.p; sz = (static_cast<size_t>(n) + 1) * sizeof(DTri); } break;
    default: return fail(RT_ERR_INVALID_ARG, "rt_gpu_debug_get_bvh: unknown selector");
    }
    if (dst) {
        if (*bytes < sz) return fail(RT_ERR_INVALID_ARG, "rt_gpu_debug_get_bvh: buffer too small");
        if (which == 0) std::memcpy(dst, src, sz);
        else if (sz) CU_CHECK(cudaMemcpy(dst, src, sz, cudaMemcpyDeviceToHost));
    }
    *bytes = sz;
    return RT_OK;
}

int rt_gpu_debug_light_pdf(rt_gpu_ctx *ctx, uint64_t n, const float *rays, float *pdf) {
    const std::string who = "rt_gpu_debug_light_pdf";
    if (!ctx || (n && (!rays || !pdf))) return fail(RT_ERR_INVALID_ARG, who + ": null argument");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, who + ": no scene uploaded");
    if (ctx->text_scene) return fail(RT_ERR_INVALID_ARG, who + ": not available for course text scenes");
    if (n > 0x7FFFFFFFu) return fail(RT_ERR_INVALID_ARG, who + ": more than 2^31 - 1 rays");
    std::fill(pdf, pdf + n, 0.0f);
    DeviceState &d = *ctx->devs[0];
    if (n == 0 || d.scene.n_lights == 0) return RT_OK;
    CU_CHECK(cudaSetDevice(d.device));
    const uint32_t m = static_cast<uint32_t>(n);
    // the rays as pending queue records: (origin, 0), (direction, pending bit)
    std::vector<float4> o4(m), d4(m);
    for (uint32_t i = 0; i < m; ++i) {
        const float *r = rays + 6 * static_cast<size_t>(i);
        o4[i] = make_float4(r[0], r[1], r[2], 0.0f);
        d4[i] = make_float4(r[3], r[4], r[5], -0.0f);  // w bits 0x80000000: pending, sample 0
    }
    struct Scratch {  // per-call buffers, freed on every return
        DevBuf<float4> o, d, o2, d2, hit;
        DevBuf<float> lpdf;
        DevBuf<uint32_t> list, slot, cnt;
        ~Scratch() {
            o.release(); d.release(); o2.release(); d2.release(); hit.release();
            lpdf.release(); list.release(); slot.release(); cnt.release();
        }
    } sb;
    if (int rc = sb.o.upload(o4, d.stream)) return rc;
    if (int rc = sb.d.upload(d4, d.stream)) return rc;
    if (int rc = sb.lpdf.alloc(m)) return rc;
    const size_t n_cnt = 8 * static_cast<size_t>(rt::kCounterStride);  // count, fetch, light_count: [2] each, own lines
    if (int rc = sb.cnt.alloc(n_cnt)) return rc;
    CU_CHECK(cudaMemsetAsync(sb.cnt.p, 0, n_cnt * sizeof(uint32_t), d.stream));
    const float inv_n_lights = 1.0f / static_cast<float>(d.scene.n_lights);
    rt::Queues q{};
    q.count = sb.cnt.p;
    q.fetch_ext = sb.cnt.p + 2 * rt::kCounterStride;
    q.fetch_shade = sb.cnt.p + 4 * rt::kCounterStride;
    q.light_count = sb.cnt.p + 6 * rt::kCounterStride;
    q.lpdf = q.lpdf_out = sb.lpdf.p;
    std::vector<float> out(m);
#if RT_EXT_WIDE8
    // k_extend8 over a queue 1 of pending rays: its light mode stores the pdf, its scene mode a hit nobody reads
    if (int rc = sb.hit.alloc(m)) return rc;
    CU_CHECK(cudaMemcpyAsync(sb.cnt.p + rt::kCounterStride, &m, sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
    q.o_in = sb.o.p;
    q.d_in = sb.d.p;
    q.hit = sb.hit.p;
    rt::k_extend8<<<d.extend_blocks, rt::kExtendThreads, 0, d.stream>>>(d.scene.scene, d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, q, 1,
                                                                         0x3F800000u);
    CU_CHECK(cudaGetLastError());
    CU_CHECK(cudaMemcpyAsync(out.data(), sb.lpdf.p, m * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaStreamSynchronize(d.stream));
    for (uint32_t i = 0; i < m; ++i) pdf[i] = out[i];
#else
    // k_shade's append (light-box test, lpdf = 0 on a miss, the list otherwise), then k_lightpdf_list as a render runs it
    if (int rc = sb.o2.alloc(m)) return rc;
    if (int rc = sb.d2.alloc(m)) return rc;
    if (int rc = sb.list.alloc(m)) return rc;
    if (int rc = sb.slot.alloc(m)) return rc;
    q.o_out = sb.o2.p;
    q.d_out = sb.d2.p;
    q.light_list = sb.list.p;
    rt::k_lightpdf_debug<<<(m + 127) / 128, 128, 0, d.stream>>>(sb.o.p, sb.d.p, m, q, d.light_box, d.scene.eps, sb.slot.p);
    CU_CHECK(cudaGetLastError());
    rt::Queues ql = q;  // queue 1 is now the input of the light kernel
    ql.o_in = sb.o2.p;
    ql.d_in = sb.d2.p;
    rt::k_lightpdf_list<<<d.light_blocks, rt::kLightThreads, 0, d.stream>>>(d.scene.light, d.scene.light_extra, inv_n_lights, d.scene.eps, ql, 1,
                                                                            0x3F800000u);
    CU_CHECK(cudaGetLastError());
    std::vector<uint32_t> slot(m);
    CU_CHECK(cudaMemcpyAsync(out.data(), sb.lpdf.p, m * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaMemcpyAsync(slot.data(), sb.slot.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream));
    CU_CHECK(cudaStreamSynchronize(d.stream));
    for (uint32_t i = 0; i < m; ++i) {
        if (slot[i] >= m) return fail(RT_ERR_CUDA, who + ": queue slot out of range");
        pdf[i] = out[slot[i]];
    }
#endif
    return RT_OK;
}

int rt_gpu_set_profiling(rt_gpu_ctx *ctx, int enable) {
    if (!ctx) return fail(RT_ERR_INVALID_ARG, "rt_gpu_set_profiling: null handle");
    ctx->profiling = enable != 0;
    return RT_OK;
}

}  // extern "C"
