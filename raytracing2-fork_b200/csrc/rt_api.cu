// rt_api.cu — the C-ABI of include/rt_b200.h: context, device memory, frame / screenshot drivers,
// multi-GPU exchange.  One ctx = one GPU; all work is enqueued on one stream (the ctx's own
// non-blocking stream or the caller's, rt_set_stream).  No exception leaves this file.
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <initializer_list>
#include <new>
#include <string>
#include <vector>

#include "rt_internal.h"

using namespace rt;

namespace {

// ---------------------------------------------------------------------------------------------- NCCL (dlopen)
// Minimal declarations of the stable NCCL C API; the library is resolved at run time so that a
// process that already carries NCCL (torch) shares its copy and a process without multi-GPU work
// never needs it.
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclUint32 = 3, ncclSum = 0 };
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
    std::string err;
};
NcclApi load_nccl() {
    NcclApi api;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) break;
    }
    if (!api.handle) {
        api.err = std::string("cannot dlopen libnccl.so.2: ") + (dlerror() ? dlerror() : "?");
        return api;
    }
    auto sym = [&](const char* s) { return dlsym(api.handle, s); };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.Reduce = (decltype(api.Reduce))sym("ncclReduce");
    api.Send = (decltype(api.Send))sym("ncclSend");
    api.Recv = (decltype(api.Recv))sym("ncclRecv");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Reduce && api.Send && api.Recv &&
             api.GroupStart && api.GroupEnd;
    if (!api.ok) api.err = "libnccl.so.2 lacks a required symbol";
    return api;
}
// function-local static: initialised exactly once, also when two threads create contexts concurrently
NcclApi& nccl() {
    static NcclApi api = load_nccl();
    return api;
}

// ---------------------------------------------------------------------------------------------- device buffers
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }  // every buffer a ctx owns goes with it: nothing to list in rt_destroy
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
        if (e == cudaSuccess) cap = bytes;
        else cudaGetLastError();  // a failed allocation is reported once (RT_ERR_OOM), not again by the next launch check
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

thread_local std::string g_static_err = "";
constexpr int kEventCap = 16384;
constexpr int kMaxBounces = 4096;

}  // namespace

struct rt_ctx {
    rt_config cfg{};
    int sm_count = 148;
    ExtendResidency extend_residency{};
    DevBuf d_query;                // the queries' [0] ray count, [1] work cursor (allocated by rt_create)
    int use_ploc = 1, shade_blocks_per_sm = 64;
    int bvh_width = 4;             // 4: k_extend walks 4-wide nodes collapsed from the binary tree; 2: the binary tree (RT_BVH_WIDTH)
    DevBuf d_wide_count;           // [0] wide nodes written, [1] worst-case traversal stack entries (k_collapse4)
    uint32_t wide_nodes = 0;
    uint32_t wide_stack_need = 0;
    uint32_t build_rounds = 0;
    int wide_depth = 0;
    bool wide_ok = false;          // 4-wide nodes built and the stack bound (3 pushes per level) holds
    int l2_max_persist = -1, l2_max_window = 0;  // device limits, -1 = not queried yet
    const void* l2_win_base = nullptr;           // the access-policy window currently set on the stream
    size_t l2_win_bytes = 0;
    uint64_t default_budget = (uint64_t)512 << 20;  // path slots in flight (128 B each = 64 GiB; capped at 40 % of the free memory)
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::string err;
    int sticky = RT_OK;

    // host copies (kept so that rt_scene_build can be repeated and for validation)
    int64_t n_tris = 0;
    int32_t n_mats = 0;
    bool built = false;
    int32_t max_mat_index = -1;
    bool tris_out_of_range = false;  // the uploaded triangles hold a NaN / inf / > 1e18 coordinate (checked at upload)
    uint32_t bvh_depth = 0;

    DevBuf d_tris, d_mats, d_tex[RT_MAX_TEXTURES];
    int tex_w[RT_MAX_TEXTURES] = {0}, tex_h[RT_MAX_TEXTURES] = {0}, tex_ch[RT_MAX_TEXTURES] = {0};
    // build scratch + outputs
    DevBuf d_centroid, d_bounds, d_keys[2], d_vals[2], d_hist, d_children, d_parent, d_boxes, d_flags, d_depth, d_node_depth;
    DevBuf d_bvh, d_grid;  // d_bvh = one arena: nodes | nodes4 | tri_geom | tri_orig | tri_shade (one L2 persisting window)
    uint4* p_nodes = nullptr;
    uint4* p_nodes4 = nullptr;   // inside the arena, right in front of the triangle records
    const void* hot_base = nullptr;  // what k_extend gathers from: [nodes4 or nodes, tri_orig end)
    cudaEvent_t build_ev[2] = {nullptr, nullptr};
    float4* p_geom = nullptr;
    float4* p_shade = nullptr;
    int32_t* p_orig = nullptr;
    size_t bvh_hot_bytes = 0;  // (wide or binary) nodes + tri_geom + tri_orig
    float grid[6] = {0, 0, 0, 1, 1, 1};
    // wavefront
    DevBuf d_path[6], d_hit, d_contrib, d_accum, d_pixrng, d_counts, d_stats, d_image, d_sum, d_out, d_rows;
    DevBuf d_stage, d_compact;  // tile-split gather
    DevBuf d_scratch[6];        // staging of host arrays (parity hooks: origins, directions, tri_id, dst, u, v)
    int width = 0, height = 0;
    std::vector<int32_t> rows;  // rows this rank owns (tile split)
    int last_frames = 0;

    // counters
    uint64_t kernel_launches = 0, extend_launches = 0;
    double build_ms = 0.0;
    std::vector<cudaEvent_t> events;
    std::vector<int> ev_tag;
    int ev_used = 0;
    double extend_ms_acc = 0.0, shade_ms_acc = 0.0;

    ncclComm_t comm = nullptr;
};

namespace {

int fail(rt_ctx* c, int code, const std::string& msg) {
    if (c) {
        c->err = msg;
        if (code == RT_ERR_CUDA || code == RT_ERR_NCCL) c->sticky = code;
    } else {
        g_static_err = msg;
    }
    return code;
}
#define CK(expr)                                                                                    \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA,           \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));                       \
    } while (0)
#define CKN(expr)                                                                                   \
    do {                                                                                            \
        ncclResult_t r__ = (expr);                                                                  \
        if (r__ != 0)                                                                               \
            return fail(ctx, RT_ERR_NCCL,                                                           \
                        std::string(#expr) + ": " +                                                 \
                            (nccl().GetErrorString ? nccl().GetErrorString(r__) : "nccl error"));   \
    } while (0)
#define GUARD()                                                                                     \
    do {                                                                                            \
        if (!ctx) return fail(nullptr, RT_ERR_INVALID, "ctx is NULL");                              \
        if (ctx->sticky != RT_OK) return ctx->sticky;                                               \
        cudaSetDevice(ctx->cfg.device);                                                             \
    } while (0)

// Does the far side of the slab test need its relative widening for rays that start at the camera?  Only when the
// origin can lie more than ~2.1 grid extents from the grid's corner (rt_scene.cuh, slab1: the rounding of the slab
// arithmetic then exceeds the builder's guard band); the bound used here is 140 000 of the 65 535 cells.
bool widen_needed(const rt_ctx* ctx, const rt_uniforms& u) {
    for (int k = 0; k < 3; k++) {
        const float r = fabsf(u.defocusDiskRight[k]) + fabsf(u.defocusDiskUp[k]);
        const float lo = (u.cameraPos[k] - r - ctx->grid[k]) * ctx->grid[3 + k];
        const float hi = (u.cameraPos[k] + r - ctx->grid[k]) * ctx->grid[3 + k];
        if (!(fabsf(lo) < 140000.0f) || !(fabsf(hi) < 140000.0f)) return true;
    }
    return false;
}

Launcher make_launcher(rt_ctx* ctx, const rt_uniforms* u = nullptr) {
    Launcher L;
    L.st = ctx->stream;
    L.widen_primary = u ? widen_needed(ctx, *u) : true;

    L.sm_count = ctx->sm_count;
    L.rng_mode = ctx->cfg.rng_mode;
    L.instrument = ctx->cfg.instrument != 0;
    L.extend_residency = &ctx->extend_residency;
    L.shade_blocks_per_sm = ctx->shade_blocks_per_sm;
    L.kernel_launches = &ctx->kernel_launches;
    L.extend_launches = &ctx->extend_launches;
    L.ev_pool = ctx->events.data();
    L.ev_cap = (int)ctx->events.size();
    L.ev_used = &ctx->ev_used;
    L.ev_tag = ctx->ev_tag.data();
    L.timing = ctx->cfg.kernel_timing != 0 && !ctx->events.empty();
    return L;
}

SceneView make_view(rt_ctx* ctx) {
    SceneView v;
    memset(&v, 0, sizeof v);
    v.nodes = ctx->p_nodes;
    v.nodes4 = ctx->wide_ok ? ctx->p_nodes4 : nullptr;
    for (int k = 0; k < 3; k++) {
        v.grid_lo[k] = ctx->grid[k];
        v.grid_inv[k] = ctx->grid[3 + k];
    }
    v.tri_geom = ctx->p_geom;
    v.tri_shade = ctx->p_shade;
    v.tri_orig = ctx->p_orig;
    v.materials = ctx->d_mats.as<float4>();
    for (int i = 0; i < RT_MAX_TEXTURES; i++) {
        v.tex_px[i] = ctx->d_tex[i].as<uint8_t>();
        v.tex_w[i] = ctx->tex_w[i];
        v.tex_h[i] = ctx->tex_h[i];
        v.tex_ch[i] = ctx->tex_ch[i];
    }
    v.num_tris = (int32_t)ctx->n_tris;
    v.num_nodes4 = (int32_t)ctx->wide_nodes;
    v.num_materials = ctx->n_mats;
    v.root_is_leaf = ctx->n_tris == 1 ? 1 : 0;
    return v;
}

// L2 persisting window over the traversal arena (nodes + triangle records): the gigabytes of path state
// that stream through every bounce should not evict the few megabytes every ray gathers from.  Measured on
// B200: no effect on config 2 (1014 ms/step with and without; the 10 MB arena stays L2-resident anyway) and
// a LOSS when the arena does not fit (config 4, 960 MB: a 10 % hitRatio window with streaming misses made
// the step 18 % slower), so the window is set only when the whole arena fits the persisting carve-out.
void apply_l2_window(rt_ctx* ctx) {
    if (!ctx->hot_base || ctx->bvh_hot_bytes == 0) return;
    if (ctx->l2_max_persist < 0) {  // device limits, queried once (cudaGetDeviceProperties costs milliseconds)
        int v = 0;
        ctx->l2_max_persist = cudaDeviceGetAttribute(&v, cudaDevAttrMaxPersistingL2CacheSize, ctx->cfg.device) == cudaSuccess ? v : 0;
        ctx->l2_max_window = cudaDeviceGetAttribute(&v, cudaDevAttrMaxAccessPolicyWindowSize, ctx->cfg.device) == cudaSuccess ? v : 0;
        cudaGetLastError();
    }
    if (ctx->l2_max_persist <= 0) return;
    const bool fits = ctx->bvh_hot_bytes <= (size_t)ctx->l2_max_persist && ctx->bvh_hot_bytes <= (size_t)ctx->l2_max_window;
    const void* base = fits ? ctx->hot_base : nullptr;
    const size_t bytes = fits ? ctx->bvh_hot_bytes : 0;
    // a rebuild of the same scene leaves the window as it is: cudaDeviceSetLimit on the persisting carve-out costs
    // tens of milliseconds of host time (measured inside bench.py's end-to-end step)
    if (base == ctx->l2_win_base && bytes == ctx->l2_win_bytes) return;
    ctx->l2_win_base = base;
    ctx->l2_win_bytes = bytes;
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof attr);  // num_bytes = 0 disables a window left by a previous, smaller scene
    if (fits) {
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes);
        attr.accessPolicyWindow.base_ptr = const_cast<void*>(ctx->hot_base);
        attr.accessPolicyWindow.num_bytes = bytes;
        attr.accessPolicyWindow.hitRatio = 1.0f;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    if (cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
}

// drain the event pool into the accumulated per-class times (stream must be idle)
void harvest_events(rt_ctx* ctx) {
    for (int i = 0; i + 1 < ctx->ev_used; i += 2) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, ctx->events[i], ctx->events[i + 1]) == cudaSuccess) {
            if (ctx->ev_tag[i] == 0) ctx->extend_ms_acc += ms; else ctx->shade_ms_acc += ms;
        }
    }
    ctx->ev_used = 0;
}

int validate_uniforms(rt_ctx* ctx, const rt_uniforms* u) {
    if (!u) return fail(ctx, RT_ERR_INVALID, "uniforms is NULL");
    if (u->width == 0 || u->height == 0 || u->width > 65536 || u->height > 65536)
        return fail(ctx, RT_ERR_INVALID, "bad image size");
    if (u->maxBounceCount > kMaxBounces) return fail(ctx, RT_ERR_INVALID, "maxBounceCount too large");
    if (u->basicShading == 0 && u->numRaysPerPixel <= 0) return fail(ctx, RT_ERR_INVALID, "numRaysPerPixel must be > 0");
    if (!ctx->built) return fail(ctx, RT_ERR_STATE, "scene not built: call rt_scene_build first");
    if (ctx->n_tris > 0 && ctx->max_mat_index >= ctx->n_mats)
        return fail(ctx, RT_ERR_STATE, "material table smaller than the scene's largest materialIndex");
    return RT_OK;
}

// (re)allocate everything that depends on the image size and the split
int prepare_image(rt_ctx* ctx, int W, int H) {
    if (W == ctx->width && H == ctx->height && !ctx->rows.empty()) return RT_OK;
    ctx->width = W;
    ctx->height = H;
    ctx->rows.clear();
    if (ctx->cfg.split_mode == RT_SPLIT_TILES && ctx->cfg.world_size > 1) {
        ctx->rows.resize((size_t)H);
        const int64_t n = rt_split_rows(H, ctx->cfg.band_rows, ctx->cfg.rank, ctx->cfg.world_size, ctx->rows.data(), H);
        ctx->rows.resize((size_t)n);
    } else {
        ctx->rows.resize((size_t)H);
        for (int y = 0; y < H; y++) ctx->rows[(size_t)y] = y;
    }
    CK(ctx->d_rows.reserve(std::max<size_t>(ctx->rows.size(), 1) * sizeof(int32_t)));
    if (!ctx->rows.empty())
        CK(cudaMemcpyAsync(ctx->d_rows.p, ctx->rows.data(), ctx->rows.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                           ctx->stream));
    CK(ctx->d_image.reserve((size_t)W * H * sizeof(float4)));
    CK(ctx->d_sum.reserve((size_t)W * H * 3 * sizeof(uint32_t)));
    CK(ctx->d_out.reserve((size_t)W * H * 3));
    CK(ctx->d_counts.reserve((size_t)(kMaxBounces + 2) * 2 * sizeof(uint32_t)));
    CK(cudaMemsetAsync(ctx->d_image.p, 0, (size_t)W * H * sizeof(float4), ctx->stream));
    return RT_OK;
}

uint64_t path_budget(rt_ctx* ctx) {
    uint64_t budget = ctx->cfg.max_paths_in_flight ? ctx->cfg.max_paths_in_flight : ctx->default_budget;
    return std::min<uint64_t>(std::max<uint64_t>(budget, 1), (uint64_t)1 << 30);  // slot ids are int32
}

// Shape of the wavefront batches for `count` frames of `spp` samples over P local pixels:
// samples of one frame in flight together, and how many frames share a batch (rt_plan_batches is the same
// arithmetic exported for tests).
void plan_batches(uint64_t budget, size_t P, int spp, int count, bool pcg, int* samples, int* frames) {
    budget = std::min<uint64_t>(std::max<uint64_t>(budget, 1), (uint64_t)1 << 30);                    // slot ids are int32
    const uint64_t perPixel = std::max<uint64_t>(budget / std::max<size_t>(P, 1), 1);  // lanes of a pixel that fit
    // the reference stream is sequential per pixel (compute.glsl:668,683): one sample of a frame at a time
    const uint64_t s = pcg ? 1 : std::min<uint64_t>(perPixel, (uint64_t)std::max(spp, 1));
    uint64_t f = 1;
    if (s == (uint64_t)std::max(spp, 1) || pcg) f = std::max<uint64_t>(perPixel / s, 1);
    *samples = (int)s;
    *frames = (int)std::min<uint64_t>(f, (uint64_t)std::max(count, 1));
}
void batch_shape(rt_ctx* ctx, size_t P, int spp, int count, int* samples, int* frames) {
    plan_batches(path_budget(ctx), P, spp, count, ctx->cfg.rng_mode == RT_RNG_REF_PCG, samples, frames);
}

int prepare_paths(rt_ctx* ctx, size_t slots, size_t frame_pixels) {
    slots = std::max<size_t>(slots, 1);
    frame_pixels = std::max<size_t>(frame_pixels, 1);
    for (int i = 0; i < 6; i++) CK(ctx->d_path[i].reserve(slots * sizeof(float4)));
    CK(ctx->d_hit.reserve(slots * sizeof(float4)));
    CK(ctx->d_contrib.reserve(slots * sizeof(float4)));
    CK(ctx->d_accum.reserve(frame_pixels * sizeof(float4)));
    CK(ctx->d_pixrng.reserve(frame_pixels * sizeof(uint32_t)));
    return RT_OK;
}

WaveBuffers make_wave(rt_ctx* ctx) {
    WaveBuffers wb;
    wb.cur = PathArrays{ctx->d_path[0].as<float4>(), ctx->d_path[1].as<float4>(), ctx->d_path[2].as<float4>()};
    wb.next = PathArrays{ctx->d_path[3].as<float4>(), ctx->d_path[4].as<float4>(), ctx->d_path[5].as<float4>()};
    wb.hit = ctx->d_hit.as<float4>();
    wb.contrib = ctx->d_contrib.as<float4>();
    wb.accum = ctx->d_accum.as<float4>();
    wb.pix_rng = ctx->d_pixrng.as<uint32_t>();
    wb.counts = ctx->d_counts.as<uint32_t>();
    wb.stats = ctx->d_stats.as<unsigned long long>();
    wb.image = ctx->d_image.as<float4>();
    wb.frame_sum = ctx->d_sum.as<uint32_t>();
    wb.out_rgb8 = ctx->d_out.as<uint8_t>();
    return wb;
}

FrameParams make_params(rt_ctx* ctx, const rt_uniforms& u) {
    FrameParams fp;
    memset(&fp, 0, sizeof fp);
    fp.u = u;
    fp.width = (int)u.width;
    fp.height = (int)u.height;
    fp.local_pixels = (int)((size_t)u.width * ctx->rows.size());
    const bool tiles = ctx->cfg.split_mode == RT_SPLIT_TILES && ctx->cfg.world_size > 1;
    fp.rows = tiles ? ctx->d_rows.as<int32_t>() : nullptr;  // identity row table = no table
    fp.div_pixels = make_fastdiv((uint32_t)fp.local_pixels);
    fp.div_samples = make_fastdiv(1u);
    fp.div_width = make_fastdiv((uint32_t)fp.width);
    fp.lanes_active = 1;
    fp.frames_in_batch = 1;
    fp.samples_in_batch = 1;
    fp.frame_stride = 1;
    fp.debug_zero_contrib = getenv("RT_DEBUG_ZERO_CONTRIB") ? 1 : 0;
    return fp;
}

// `count` frames with frameIndex = first, first + stride, …, each numRaysPerPixel samples per local pixel,
// resolved into the image (+ the 8-bit sums).  Frames are batched together when they fit the path budget.
int render_frames(rt_ctx* ctx, const rt_uniforms& u, uint32_t first, int stride, int count, bool add_to_sum) {
    const int W = (int)u.width, H = (int)u.height;
    int rc = prepare_image(ctx, W, H);
    if (rc) return rc;
    Launcher L = make_launcher(ctx, &u);
    SceneView sc = make_view(ctx);
    FrameParams fp = make_params(ctx, u);
    if (fp.local_pixels == 0 || count <= 0) return RT_OK;
    if (u.basicShading != 0) {
        WaveBuffers wb = make_wave(ctx);
        fp.u.frameIndex = first + (uint32_t)((count - 1) * stride);
        CK(wf_preview(L, sc, wb, fp));
        return RT_OK;
    }
    const int spp = u.numRaysPerPixel;
    const size_t P = (size_t)fp.local_pixels;
    int samples = 1, framesPerBatch = 1;
    batch_shape(ctx, P, spp, count, &samples, &framesPerBatch);
    rc = prepare_paths(ctx, P * samples * framesPerBatch, P * framesPerBatch);
    if (rc) return rc;
    WaveBuffers wb = make_wave(ctx);
    fp.frame_stride = stride;
    for (int done = 0; done < count; done += framesPerBatch) {
        fp.u.frameIndex = first + (uint32_t)(done * stride);  // rayTracing.cpp:187
        fp.frames_in_batch = std::min(framesPerBatch, count - done);
        CK(wf_clear_accum(L, wb, (long long)P * fp.frames_in_batch));
        if (ctx->cfg.rng_mode == RT_RNG_REF_PCG) CK(wf_seed_pixels(L, sc, wb, fp));
        for (int base = 0; base < spp; base += samples) {
            fp.sample_base = base;
            fp.samples_in_batch = std::min(samples, spp - base);
            fp.div_samples = make_fastdiv((uint32_t)fp.samples_in_batch);
            fp.lanes_active = fp.frames_in_batch * fp.samples_in_batch;
            CK(wf_render_batch(L, sc, wb, fp));
        }
        CK(wf_resolve_frame(L, wb, fp, add_to_sum));
        // keep the event pool from overflowing on long screenshots
        if (ctx->cfg.kernel_timing && ctx->ev_used > kEventCap - 512) {
            CK(cudaStreamSynchronize(ctx->stream));
            harvest_events(ctx);
        }
    }
    return RT_OK;
}

int render_one_frame(rt_ctx* ctx, const rt_uniforms& u, bool add_to_sum) {
    return render_frames(ctx, u, u.frameIndex, 1, 1, add_to_sum);
}

// partial sums of the frames (or rows) this rank owns, left in d_sum
int render_partial(rt_ctx* ctx, const rt_uniforms* uniforms, int frames) {
    int rc = validate_uniforms(ctx, uniforms);
    if (rc) return rc;
    if (frames <= 0) return fail(ctx, RT_ERR_INVALID, "frames must be > 0");
    const int W = (int)uniforms->width, H = (int)uniforms->height;
    rc = prepare_image(ctx, W, H);
    if (rc) return rc;
    CK(cudaMemsetAsync(ctx->d_sum.p, 0, (size_t)W * H * 3 * sizeof(uint32_t), ctx->stream));
    const bool frameSplit = ctx->cfg.split_mode == RT_SPLIT_FRAMES && ctx->cfg.world_size > 1;
    rt_uniforms uf = *uniforms;
    uf.basicShading = 0;  // rayTracing.cpp:146 (SCREENSHOT_BASIC_SHADING)
    // frame f carries frameIndex = f (rayTracing.cpp:187); under RT_SPLIT_FRAMES this rank owns f % world == rank
    const int first = frameSplit ? ctx->cfg.rank : 0;
    const int stride = frameSplit ? ctx->cfg.world_size : 1;
    const int count = first < frames ? (frames - first + stride - 1) / stride : 0;
    rc = render_frames(ctx, uf, (uint32_t)first, stride, count, true);
    if (rc) return rc;
    ctx->last_frames = frames;
    return RT_OK;
}

// bring every rank's partial sums to rank 0 (d_sum of rank 0 holds the total afterwards)
int exchange_partials(rt_ctx* ctx) {
    if (ctx->cfg.world_size <= 1 || ctx->cfg.split_mode == RT_SPLIT_NONE) return RT_OK;
    if (!ctx->comm) return fail(ctx, RT_ERR_STATE, "world_size > 1 but rt_comm_init was not called");
    NcclApi& N = nccl();
    const int W = ctx->width, H = ctx->height;
    const size_t count = (size_t)W * H * 3;
    if (ctx->cfg.split_mode == RT_SPLIT_FRAMES) {
        // sums of 8-bit integers: exact in u32, so the total is independent of the GPU count
        CKN(N.Reduce(ctx->d_sum.p, ctx->d_sum.p, count, ncclUint32, ncclSum, 0, ctx->comm, ctx->stream));
        return RT_OK;
    }
    // RT_SPLIT_TILES: a gather, not a reduce — each rank ships only the rows it rendered
    Launcher L = make_launcher(ctx);
    const size_t rowLen = (size_t)W * 3;
    if (ctx->cfg.rank != 0) {
        CK(ctx->d_compact.reserve(std::max<size_t>(ctx->rows.size() * rowLen, 1) * sizeof(uint32_t)));
        CK(wf_gather_rows(L, ctx->d_sum.as<uint32_t>(), ctx->d_compact.as<uint32_t>(), ctx->d_rows.as<int32_t>(),
                          (int)ctx->rows.size(), W));
        if (!ctx->rows.empty())
            CKN(N.Send(ctx->d_compact.p, ctx->rows.size() * rowLen, ncclUint32, 0, ctx->comm, ctx->stream));
        return RT_OK;
    }
    std::vector<std::vector<int32_t>> peerRows((size_t)ctx->cfg.world_size);
    size_t total = 0;
    for (int r = 1; r < ctx->cfg.world_size; r++) {
        peerRows[(size_t)r].resize((size_t)H);
        const int64_t n = rt_split_rows(H, ctx->cfg.band_rows, r, ctx->cfg.world_size, peerRows[(size_t)r].data(), H);
        peerRows[(size_t)r].resize((size_t)n);
        total += (size_t)n;
    }
    CK(ctx->d_stage.reserve(std::max<size_t>(total * rowLen, 1) * sizeof(uint32_t)));
    CK(ctx->d_compact.reserve(std::max<size_t>(total, 1) * sizeof(int32_t)));
    std::vector<int32_t> allRows;
    for (int r = 1; r < ctx->cfg.world_size; r++) allRows.insert(allRows.end(), peerRows[(size_t)r].begin(), peerRows[(size_t)r].end());
    if (total) CK(cudaMemcpyAsync(ctx->d_compact.p, allRows.data(), total * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CKN(N.GroupStart());
    size_t off = 0;
    for (int r = 1; r < ctx->cfg.world_size; r++) {
        const size_t n = peerRows[(size_t)r].size();
        if (n) CKN(N.Recv(ctx->d_stage.as<uint32_t>() + off * rowLen, n * rowLen, ncclUint32, r, ctx->comm, ctx->stream));
        off += n;
    }
    CKN(N.GroupEnd());
    CK(wf_scatter_rows(L, ctx->d_stage.as<uint32_t>(), ctx->d_sum.as<uint32_t>(), ctx->d_compact.as<int32_t>(), (int)total, W));
    CK(cudaStreamSynchronize(ctx->stream));  // allRows must outlive the async copy
    return RT_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

const char* rt_version(void) { return "rt_b200 0.1 (sm_100a)"; }

const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_static_err.c_str(); }

int rt_create(rt_ctx** out, const rt_config* cfg) {
    if (!out || !cfg) return fail(nullptr, RT_ERR_INVALID, "rt_create: NULL argument");
    *out = nullptr;
    if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size)
        return fail(nullptr, RT_ERR_INVALID, "rt_create: bad rank / world_size");
    if (cfg->rng_mode != RT_RNG_REF_PCG && cfg->rng_mode != RT_RNG_PHILOX)
        return fail(nullptr, RT_ERR_INVALID, "rt_create: bad rng_mode");
    if (cfg->split_mode < RT_SPLIT_NONE || cfg->split_mode > RT_SPLIT_FRAMES)
        return fail(nullptr, RT_ERR_INVALID, "rt_create: bad split_mode");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0)
        return fail(nullptr, RT_ERR_NO_DEVICE,
                    std::string("rt_create: no CUDA device (this backend has no CPU fallback): ") + cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, RT_ERR_INVALID, "rt_create: bad device ordinal");
    rt_ctx* ctx = new (std::nothrow) rt_ctx;
    if (!ctx) return fail(nullptr, RT_ERR_OOM, "rt_create: out of host memory");
    ctx->cfg = *cfg;
    cudaSetDevice(cfg->device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    // fails only when the library has no image this device can load, which every launch would report too
    e = wf_extend_residency(cfg->instrument != 0, &ctx->extend_residency);
    if (e != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ERR_CUDA, std::string("rt_create: k_extend occupancy: ") + cudaGetErrorString(e));
    }
    e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        std::string m = std::string("rt_create: cudaStreamCreate: ") + cudaGetErrorString(e);
        delete ctx;
        return fail(nullptr, RT_ERR_CUDA, m);
    }
    ctx->stream = ctx->own_stream;
    {
        // Path slots: fewer, larger wavefronts amortise the drain of the persistent kernels (config 2: 8 lanes
        // per pixel 1203 ms/step, 64 lanes 1057 ms; round 2: 128 Mi slots 744.8 ms, 512 Mi — the whole 4-frame
        // screenshot in one wavefront, a 4K frame in one — 735.5 ms).  HBM is there to be used: default 512 Mi slots
        // = 64 GiB, never more than 40 % of what is free, and only what a job needs is ever allocated.
        size_t freeB = 0, totalB = 0;
        if (cudaMemGetInfo(&freeB, &totalB) == cudaSuccess && freeB > 0)
            ctx->default_budget = std::min<uint64_t>(ctx->default_budget, (uint64_t)(freeB * 0.4) / 128u);
        if (ctx->default_budget < (1u << 20)) ctx->default_budget = 1u << 20;
    }
    // switches that keep the fallback and test-only paths reachable (README)
    if (const char* e9 = getenv("RT_SHADE_BLOCKS_PER_SM")) ctx->shade_blocks_per_sm = std::max(1, std::min(256, atoi(e9)));
    if (const char* e8 = getenv("RT_MAX_PATHS_MI")) ctx->default_budget = (uint64_t)std::max(1, atoi(e8)) << 20;
    if (const char* e9 = getenv("RT_BVH_WIDTH")) ctx->bvh_width = atoi(e9) == 4 ? 4 : 2;
    if (const char* e5 = getenv("RT_BVH_BUILDER")) ctx->use_ploc = strcmp(e5, "lbvh") != 0;
    if (ctx->d_stats.reserve(4 * sizeof(unsigned long long)) != cudaSuccess ||
        cudaMemsetAsync(ctx->d_stats.p, 0, 4 * sizeof(unsigned long long), ctx->stream) != cudaSuccess ||
        ctx->d_query.reserve(2 * sizeof(uint32_t)) != cudaSuccess) {
        delete ctx;
        return fail(nullptr, RT_ERR_CUDA, "rt_create: cannot allocate counters");
    }
    if (cfg->kernel_timing) {
        ctx->events.resize(kEventCap);
        ctx->ev_tag.resize(kEventCap);
        for (auto& ev : ctx->events) cudaEventCreate(&ev);
    }
    *out = ctx;
    return RT_OK;
}

void rt_destroy(rt_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && nccl().ok) nccl().CommDestroy(ctx->comm);
    for (auto& ev : ctx->events) cudaEventDestroy(ev);
    for (auto& ev : ctx->build_ev) if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;  // ~DevBuf releases every device buffer
}

int rt_set_stream(rt_ctx* ctx, void* cuda_stream) {
    GUARD();
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->l2_win_base) {  // the window is a per-stream attribute: do not leave ours on a stream we hand back
        cudaStreamAttrValue attr;
        memset(&attr, 0, sizeof attr);
        if (cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
    }
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    ctx->l2_win_base = nullptr;
    ctx->l2_win_bytes = 0;
    apply_l2_window(ctx);
    return RT_OK;
}

int rt_scene_set_triangles(rt_ctx* ctx, const rt_triangle* tris, int64_t count) {
    GUARD();
    if (count < 0 || (count > 0 && !tris)) return fail(ctx, RT_ERR_INVALID, "rt_scene_set_triangles: bad argument");
    if (count > (int64_t)kLeafFirstMask - 8) return fail(ctx, RT_ERR_INVALID, "rt_scene_set_triangles: more than 2^27-9 triangles");
    // validate on the host copy the caller still owns, BEFORE any state of the ctx changes: a rejected call
    // leaves the previous scene (and its max_mat_index) exactly as it was
    int32_t maxMat = -1, minMat = 0;
    for (int64_t i = 0; i < count; i++) {
        maxMat = std::max(maxMat, tris[i].materialIndex);
        minMat = std::min(minMat, tris[i].materialIndex);
    }
    if (minMat < 0) return fail(ctx, RT_ERR_INVALID, "rt_scene_set_triangles: negative materialIndex");
    ctx->built = false;  // from here on the old scene is gone, whatever happens
    ctx->n_tris = 0;
    ctx->max_mat_index = -1;
    CK(ctx->d_tris.reserve(std::max<size_t>((size_t)count, 1) * sizeof(rt_triangle)));
    if (count) CK(cudaMemcpyAsync(ctx->d_tris.p, tris, (size_t)count * sizeof(rt_triangle), cudaMemcpyHostToDevice, ctx->stream));
    // coordinate range check on the device copy (one pass at HBM speed), read back with the sync the upload needs anyway
    uint32_t outOfRange = 0;
    CK(ctx->d_depth.reserve(kBuildStatusWords * sizeof(uint32_t)));
    CK(validate_triangles(ctx->d_tris.as<rt_triangle>(), (int)count, ctx->d_depth.as<uint32_t>(), ctx->sm_count, ctx->stream));
    CK(cudaMemcpyAsync(&outOfRange, ctx->d_depth.p, sizeof outOfRange, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // glBufferData semantics: the caller may free at once
    ctx->n_tris = count;
    ctx->max_mat_index = maxMat;
    ctx->tris_out_of_range = outOfRange != 0;
    return RT_OK;
}

int rt_scene_set_materials(rt_ctx* ctx, const rt_material* mats, int32_t count) {
    GUARD();
    if (count <= 0 || !mats) return fail(ctx, RT_ERR_INVALID, "rt_scene_set_materials: bad argument");
    // a built scene keeps rendering with the new table only if every triangle still finds its material
    if (ctx->built && ctx->n_tris > 0 && ctx->max_mat_index >= count)
        return fail(ctx, RT_ERR_INVALID, "rt_scene_set_materials: the built scene references material " +
                                             std::to_string(ctx->max_mat_index) + ", table has " + std::to_string(count));
    CK(cudaStreamSynchronize(ctx->stream));  // frames in flight still read the old table
    CK(ctx->d_mats.reserve((size_t)count * sizeof(rt_material)));
    CK(cudaMemcpyAsync(ctx->d_mats.p, mats, (size_t)count * sizeof(rt_material), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_mats = count;
    return RT_OK;
}

int rt_scene_set_texture(rt_ctx* ctx, int32_t slot, const uint8_t* pixels, int32_t w, int32_t h, int32_t ch) {
    GUARD();
    if (slot < 0 || slot >= RT_MAX_TEXTURES || !pixels || w <= 0 || h <= 0 || ch < 1 || ch > 4)
        return fail(ctx, RT_ERR_INVALID, "rt_scene_set_texture: bad argument");
    const size_t bytes = (size_t)w * h * ch;
    CK(ctx->d_tex[slot].reserve(bytes));
    CK(cudaMemcpyAsync(ctx->d_tex[slot].p, pixels, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->tex_w[slot] = w;
    ctx->tex_h[slot] = h;
    ctx->tex_ch[slot] = ch;
    return RT_OK;
}

int rt_scene_build(rt_ctx* ctx) {
    GUARD();
    if (ctx->n_mats <= 0) return fail(ctx, RT_ERR_STATE, "rt_scene_build: no materials");
    if (ctx->n_tris > 0 && ctx->max_mat_index >= ctx->n_mats)
        return fail(ctx, RT_ERR_INVALID, "rt_scene_build: a triangle's materialIndex is out of range");
    const int n = (int)ctx->n_tris;
    ctx->built = false;
    ctx->wide_ok = false;
    if (ctx->tris_out_of_range)  // not sticky: upload a finite scene and build again
        return fail(ctx, RT_ERR_INVALID, "rt_scene_build: a triangle has a non-finite vertex coordinate (NaN, inf or |x| > 1e18)");
    if (n == 0) {
        ctx->built = true;
        ctx->bvh_depth = 0;
        return RT_OK;
    }
    const size_t nn = (size_t)std::max(n - 1, 1);
    const bool wantWide = ctx->bvh_width == 4 && n >= 2;
    CK(ctx->d_centroid.reserve((size_t)n * sizeof(float4)));
    CK(ctx->d_bounds.reserve(12 * sizeof(uint32_t)));
    for (int i = 0; i < 2; i++) {
        CK(ctx->d_keys[i].reserve((size_t)n * sizeof(uint64_t)));
        CK(ctx->d_vals[i].reserve((size_t)n * sizeof(uint32_t)));
    }
    CK(ctx->d_hist.reserve(build_scratch_words(n) * sizeof(uint32_t)));
    CK(ctx->d_children.reserve(2 * nn * sizeof(int32_t)));
    CK(ctx->d_parent.reserve((size_t)(2 * n) * sizeof(int32_t)));
    CK(ctx->d_boxes.reserve((size_t)(2 * n) * 2 * sizeof(float4)));
    CK(ctx->d_flags.reserve(((size_t)n + 1) * sizeof(uint32_t)));
    CK(ctx->d_node_depth.reserve((size_t)(2 * n) * sizeof(uint32_t)));
    CK(ctx->d_depth.reserve(kBuildStatusWords * sizeof(uint32_t)));
    CK(ctx->d_grid.reserve(6 * sizeof(float)));
    CK(ctx->d_wide_count.reserve(2 * sizeof(uint32_t)));
    {
        // one arena, in the order the traversal touches it: binary nodes (preview, RT_BVH_WIDTH=2) | 4-wide
        // nodes | triangle records | original indices | shading records.  The L2 persisting window covers what
        // k_extend gathers from: [wide nodes (or binary nodes when there are none), end of the original indices).
        auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t bNodes = up(nn * 2 * sizeof(uint4)), bNodes4 = wantWide ? up(nn * 4 * sizeof(uint4)) : 0,
                     bGeom = up((size_t)n * 4 * sizeof(float4)), bOrig = up((size_t)n * sizeof(int32_t)),
                     bShade = up((size_t)n * 2 * sizeof(float4));
        CK(ctx->d_bvh.reserve(bNodes + bNodes4 + bGeom + bOrig + bShade));
        char* base = ctx->d_bvh.as<char>();
        ctx->p_nodes = reinterpret_cast<uint4*>(base);
        ctx->p_nodes4 = wantWide ? reinterpret_cast<uint4*>(base + bNodes) : nullptr;
        ctx->p_geom = reinterpret_cast<float4*>(base + bNodes + bNodes4);
        ctx->p_orig = reinterpret_cast<int32_t*>(base + bNodes + bNodes4 + bGeom);
        ctx->p_shade = reinterpret_cast<float4*>(base + bNodes + bNodes4 + bGeom + bOrig);
        ctx->hot_base = wantWide ? (const void*)ctx->p_nodes4 : (const void*)ctx->p_nodes;
        ctx->bvh_hot_bytes = (wantWide ? bNodes4 : bNodes) + bGeom + bOrig;
    }
    BuildArgs a;
    a.tris = ctx->d_tris.as<rt_triangle>();
    a.n = n;
    a.use_ploc = ctx->use_ploc;
    a.centroid = ctx->d_centroid.as<float4>();
    a.bounds = ctx->d_bounds.as<uint32_t>();
    for (int i = 0; i < 2; i++) {
        a.keys[i] = ctx->d_keys[i].as<uint64_t>();
        a.vals[i] = ctx->d_vals[i].as<uint32_t>();
    }
    a.hist = ctx->d_hist.as<uint32_t>();
    a.children = ctx->d_children.as<int32_t>();
    a.parent = ctx->d_parent.as<int32_t>();
    a.boxes = ctx->d_boxes.as<float4>();
    a.flags = ctx->d_flags.as<uint32_t>();
    a.nodeDepth = ctx->d_node_depth.as<uint32_t>();
    a.status = ctx->d_depth.as<uint32_t>();
    a.nodes = ctx->p_nodes;
    a.nodes4 = ctx->p_nodes4;
    a.wide_count = wantWide ? ctx->d_wide_count.as<uint32_t>() : nullptr;
    int wideLevels = 0;
    a.wide_levels = &wideLevels;
    a.grid = ctx->d_grid.as<float>();
    a.geom = ctx->p_geom;
    a.shade = ctx->p_shade;
    a.orig = ctx->p_orig;
    a.sm_count = ctx->sm_count;
    for (auto& ev : ctx->build_ev)
        if (!ev) CK(cudaEventCreate(&ev));
    uint32_t status[kBuildStatusWords] = {0};
    uint32_t wide[2] = {0, 0};
    auto run = [&]() -> int {
        CK(cudaEventRecord(ctx->build_ev[0], ctx->stream));
        CK(build_lbvh(a, ctx->stream, &ctx->kernel_launches));
        CK(cudaEventRecord(ctx->build_ev[1], ctx->stream));
        CK(cudaMemcpyAsync(status, ctx->d_depth.p, sizeof status, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(ctx->grid, ctx->d_grid.p, sizeof ctx->grid, cudaMemcpyDeviceToHost, ctx->stream));
        if (a.wide_count) CK(cudaMemcpyAsync(wide, a.wide_count, sizeof wide, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    };
    int rc = run();
    if (rc) return rc;
    if (status[kBuildNonFinite])
        return fail(ctx, RT_ERR_INVALID, "rt_scene_build: a triangle has a non-finite vertex coordinate");
    if (a.use_ploc && (status[kBuildPlocStuck] || (int)status[kBuildDepth] + 1 >= kStackSize)) {
        // agglomerative clustering can chain (one big cluster absorbing neighbours round after round) or, with
        // boxes whose union area overflows, find no mutual pair at all; the Karras tree over the same Morton
        // order is at most key-bits deep and always exists
        a.use_ploc = 0;
        rc = run();
        if (rc) return rc;
    }
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, ctx->build_ev[0], ctx->build_ev[1]);
    ctx->build_ms = ms;
    ctx->bvh_depth = status[kBuildDepth];
    ctx->build_rounds = a.use_ploc ? status[kBuildPlocRounds] : 0u;
    if ((int)ctx->bvh_depth + 1 >= kStackSize)
        return fail(ctx, RT_ERR_INVALID, "rt_scene_build: BVH deeper than the traversal stack (" + std::to_string(ctx->bvh_depth) + ")");
    // a 4-wide visit pushes at most (children - 1) entries; k_collapse4 tracks the worst root-to-leaf total
    ctx->wide_nodes = wide[0];
    ctx->wide_stack_need = wide[1];
    ctx->wide_ok = a.nodes4 != nullptr && wideLevels > 0 && (int)wide[1] + 2 < kStackSize;
    ctx->wide_depth = wideLevels;
    ctx->built = true;
    apply_l2_window(ctx);
    return RT_OK;
}

int rt_render_frame(rt_ctx* ctx, const rt_uniforms* uniforms) {
    GUARD();
    int rc = validate_uniforms(ctx, uniforms);
    if (rc) return rc;
    return render_one_frame(ctx, *uniforms, false);
}

int rt_read_frame_rgba32f(rt_ctx* ctx, float* dst) {
    GUARD();
    if (!dst || ctx->width == 0) return fail(ctx, RT_ERR_INVALID, "rt_read_frame_rgba32f: nothing rendered / NULL dst");
    CK(cudaMemcpyAsync(dst, ctx->d_image.p, (size_t)ctx->width * ctx->height * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_screenshot_partial(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames) {
    GUARD();
    return render_partial(ctx, uniforms, frames);
}

int rt_read_frame_sum(rt_ctx* ctx, uint32_t* dst) {
    GUARD();
    if (!dst || ctx->width == 0) return fail(ctx, RT_ERR_INVALID, "rt_read_frame_sum: nothing rendered / NULL dst");
    CK(cudaMemcpyAsync(dst, ctx->d_sum.p, (size_t)ctx->width * ctx->height * 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_finalize_sums(rt_ctx* ctx, const uint32_t* sums, int32_t width, int32_t height, int32_t frames, uint8_t* rgb8) {
    GUARD();
    if (!sums || !rgb8 || width <= 0 || height <= 0 || frames <= 0) return fail(ctx, RT_ERR_INVALID, "rt_finalize_sums: bad argument");
    const size_t count = (size_t)width * height * 3;
    CK(ctx->d_scratch[0].reserve(count * sizeof(uint32_t)));
    CK(ctx->d_scratch[1].reserve(count));
    CK(cudaMemcpyAsync(ctx->d_scratch[0].p, sums, count * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    Launcher L = make_launcher(ctx);
    CK(wf_finalize(L, ctx->d_scratch[0].as<uint32_t>(), ctx->d_scratch[1].as<uint8_t>(), width, height, frames));
    CK(cudaMemcpyAsync(rgb8, ctx->d_scratch[1].p, count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_screenshot_device(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames) {
    GUARD();
    int rc = render_partial(ctx, uniforms, frames);
    if (rc) return rc;
    rc = exchange_partials(ctx);
    if (rc) return rc;
    if (ctx->cfg.rank == 0) {
        Launcher L = make_launcher(ctx);
        CK(wf_finalize(L, ctx->d_sum.as<uint32_t>(), ctx->d_out.as<uint8_t>(), ctx->width, ctx->height, frames));
    }
    return RT_OK;
}

int rt_screenshot_fetch(rt_ctx* ctx, uint8_t* rgb8) {
    GUARD();
    if (ctx->width == 0) return fail(ctx, RT_ERR_STATE, "rt_screenshot_fetch: nothing rendered");
    if (ctx->cfg.rank == 0) {
        if (!rgb8) return fail(ctx, RT_ERR_INVALID, "rt_screenshot_fetch: NULL destination on rank 0");
        CK(cudaMemcpyAsync(rgb8, ctx->d_out.p, (size_t)ctx->width * ctx->height * 3, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_screenshot(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames, uint8_t* rgb8) {
    int rc = rt_screenshot_device(ctx, uniforms, frames);
    if (rc) return rc;
    return rt_screenshot_fetch(ctx, rgb8);
}

namespace {
// Closest hit of n rays whose (N, 3) origins and directions are in device memory: k_extend's CLOSEST query, on the ctx
// stream, with the ctx's count and cursor words.  rt_query_closest passes the caller's arrays, the parity hooks
// their staged copies and no tmax.
int closest_query(rt_ctx* ctx, const float* o3, const float* d3, const float* tmax, int64_t n, int32_t* tri,
                  float* dst, float* bu, float* bv) {
    const QueryArgs q{o3, d3, tmax, tri, dst, bu, bv, nullptr};
    CK(wf_query(make_launcher(ctx), make_view(ctx), q, n, Query::CLOSEST, ctx->d_query.as<uint32_t>(),
                ctx->d_stats.as<unsigned long long>()));
    return RT_OK;
}
}  // namespace

int rt_first_hit(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t mode, int32_t* tri_id, float* dst) {
    GUARD();
    int rc = validate_uniforms(ctx, uniforms);
    if (rc) return rc;
    if (mode != RT_FIRST_HIT_CENTRE && mode != RT_FIRST_HIT_SAMPLE0) return fail(ctx, RT_ERR_INVALID, "rt_first_hit: bad mode");
    const size_t n = (size_t)uniforms->width * uniforms->height;
    CK(ctx->d_scratch[0].reserve(n * 3 * sizeof(float)));
    CK(ctx->d_scratch[1].reserve(n * 3 * sizeof(float)));
    CK(ctx->d_scratch[2].reserve(n * sizeof(int32_t)));
    CK(ctx->d_scratch[3].reserve(n * sizeof(float)));
    FrameParams fp;
    memset(&fp, 0, sizeof fp);
    fp.u = *uniforms;
    fp.width = (int)uniforms->width;
    fp.height = (int)uniforms->height;
    CK(wf_first_rays(make_launcher(ctx), fp, mode, ctx->d_scratch[0].as<float>(), ctx->d_scratch[1].as<float>()));
    rc = closest_query(ctx, ctx->d_scratch[0].as<float>(), ctx->d_scratch[1].as<float>(), nullptr, (int64_t)n,
                       ctx->d_scratch[2].as<int32_t>(), ctx->d_scratch[3].as<float>(), nullptr, nullptr);
    if (rc) return rc;
    if (tri_id) CK(cudaMemcpyAsync(tri_id, ctx->d_scratch[2].p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (dst) CK(cudaMemcpyAsync(dst, ctx->d_scratch[3].p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_trace_rays(rt_ctx* ctx, const float* origins, const float* dirs, int64_t count, int32_t* tri_id, float* dst,
                  float* bu, float* bv) {
    GUARD();
    if (!ctx->built) return fail(ctx, RT_ERR_STATE, "scene not built: call rt_scene_build first");
    if (count < 0 || (count > 0 && (!origins || !dirs))) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays: bad argument");
    if (count == 0) return RT_OK;
    if (count > ((int64_t)1 << 30)) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays: more than 2^30 rays in one call");
    const size_t n = (size_t)count;
    CK(ctx->d_scratch[0].reserve(n * 3 * sizeof(float)));
    CK(ctx->d_scratch[1].reserve(n * 3 * sizeof(float)));
    for (int i = 2; i < 6; i++) CK(ctx->d_scratch[i].reserve(n * sizeof(float)));
    CK(cudaMemcpyAsync(ctx->d_scratch[0].p, origins, n * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_scratch[1].p, dirs, n * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    const int rc = closest_query(ctx, ctx->d_scratch[0].as<float>(), ctx->d_scratch[1].as<float>(), nullptr, count,
                                 ctx->d_scratch[2].as<int32_t>(), ctx->d_scratch[3].as<float>(),
                                 ctx->d_scratch[4].as<float>(), ctx->d_scratch[5].as<float>());
    if (rc) return rc;
    if (tri_id) CK(cudaMemcpyAsync(tri_id, ctx->d_scratch[2].p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (dst) CK(cudaMemcpyAsync(dst, ctx->d_scratch[3].p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (bu) CK(cudaMemcpyAsync(bu, ctx->d_scratch[4].p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (bv) CK(cudaMemcpyAsync(bv, ctx->d_scratch[5].p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

namespace {
// Everything a query checks before it enqueues anything.  `inputs` (named `what`) must not be NULL, `bound` (tmax or
// max_dist) may be.  The arrays must be device (or managed) memory of the ctx's device: the kernels read and write
// them in place.
int validate_query(rt_ctx* ctx, const char* fn, const char* what, std::initializer_list<const float*> inputs,
                   const float* bound, int64_t count, std::initializer_list<const void*> outputs) {
    if (!ctx->built) return fail(ctx, RT_ERR_STATE, "scene not built: call rt_scene_build first");
    if (count < 0) return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": count < 0");
    if (count > ((int64_t)1 << 30)) return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": more than 2^30 queries in one call");
    if (count == 0) return RT_OK;
    for (const float* p : inputs)
        if (!p) return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": NULL " + what);
    auto on_device = [&](const void* p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == ctx->cfg.device;
    };
    bool inputs_ok = !bound || on_device(bound);
    for (const float* p : inputs) inputs_ok = inputs_ok && on_device(p);
    if (!inputs_ok)
        return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": an input is not device memory of device " +
                                             std::to_string(ctx->cfg.device));
    for (const void* p : outputs)
        if (p && !on_device(p))
            return fail(ctx, RT_ERR_INVALID, std::string(fn) + ": an output is not device memory of device " +
                                                 std::to_string(ctx->cfg.device));
    return RT_OK;
}
}  // namespace

int rt_query_closest(rt_ctx* ctx, const float* origins, const float* dirs, const float* tmax, int64_t count,
                     int32_t* tri_id, float* dst, float* bu, float* bv) {
    GUARD();
    int rc = validate_query(ctx, "rt_query_closest", "origins or dirs", {origins, dirs}, tmax, count, {tri_id, dst, bu, bv});
    if (rc || count == 0) return rc;
    return closest_query(ctx, origins, dirs, tmax, count, tri_id, dst, bu, bv);
}

int rt_query_occluded(rt_ctx* ctx, const float* origins, const float* dirs, const float* tmax, int64_t count,
                      uint8_t* occluded) {
    GUARD();
    if (count > 0 && !occluded) return fail(ctx, RT_ERR_INVALID, "rt_query_occluded: NULL occluded");
    int rc = validate_query(ctx, "rt_query_occluded", "origins or dirs", {origins, dirs}, tmax, count, {occluded});
    if (rc || count == 0) return rc;
    const QueryArgs q{origins, dirs, tmax, nullptr, nullptr, nullptr, nullptr, occluded};
    CK(wf_query(make_launcher(ctx), make_view(ctx), q, count, Query::ANY, ctx->d_query.as<uint32_t>(),
                ctx->d_stats.as<unsigned long long>()));
    return RT_OK;
}

int rt_query_nearest(rt_ctx* ctx, const float* points, const float* max_dist, int64_t count, int32_t* tri_id,
                     float* dist, float* bu, float* bv, float* closest) {
    GUARD();
    int rc = validate_query(ctx, "rt_query_nearest", "points", {points}, max_dist, count, {tri_id, dist, bu, bv, closest});
    if (rc || count == 0) return rc;
    const NearestArgs q{points, max_dist, tri_id, dist, bu, bv, closest};
    CK(wf_nearest(make_launcher(ctx), make_view(ctx), q, count, ctx->d_stats.as<unsigned long long>()));
    return RT_OK;
}

int rt_scene_get_bvh(rt_ctx* ctx, rt_bvh_node* nodes, int64_t* node_count, int32_t* sorted_tri_ids, int64_t* tri_count,
                     float scene_lo[3], float scene_hi[3]) {
    GUARD();
    if (!ctx->built) return fail(ctx, RT_ERR_STATE, "scene not built");
    const int64_t n = ctx->n_tris;
    const int64_t nn = n >= 2 ? n - 1 : 0;
    if (node_count) *node_count = nn;
    if (tri_count) *tri_count = n;
    CK(cudaStreamSynchronize(ctx->stream));
    if (nodes && nn > 0) {
        std::vector<uint4> raw((size_t)nn * 2);
        CK(cudaMemcpy(raw.data(), ctx->p_nodes, raw.size() * sizeof(uint4), cudaMemcpyDeviceToHost));
        const float* G = ctx->grid;
        auto deq = [&](uint32_t q, int k) { return G[k] + (float)q / G[3 + k]; };
        for (int64_t i = 0; i < nn; i++) {
            const uint4 a = raw[(size_t)i * 2], b = raw[(size_t)i * 2 + 1];
            rt_bvh_node& o = nodes[i];
            // one word per axis: lower plane | extent << 16
            auto hiq = [](uint32_t w) { return (w & 0xffffu) + (w >> 16); };
            o.lo_x[0] = deq(a.x & 0xffffu, 0); o.hi_x[0] = deq(hiq(a.x), 0);
            o.lo_y[0] = deq(a.y & 0xffffu, 1); o.hi_y[0] = deq(hiq(a.y), 1);
            o.lo_z[0] = deq(a.z & 0xffffu, 2); o.hi_z[0] = deq(hiq(a.z), 2);
            o.lo_x[1] = deq(a.w & 0xffffu, 0); o.hi_x[1] = deq(hiq(a.w), 0);
            o.lo_y[1] = deq(b.x & 0xffffu, 1); o.hi_y[1] = deq(hiq(b.x), 1);
            o.lo_z[1] = deq(b.y & 0xffffu, 2); o.hi_z[1] = deq(hiq(b.y), 2);
            const int32_t c[2] = {(int32_t)b.z, (int32_t)b.w};
            for (int k = 0; k < 2; k++) {
                if (c[k] >= 0) {
                    o.child[k] = c[k];
                    o.count[k] = 0;
                } else {
                    const int32_t packed = ~c[k];
                    o.child[k] = ~(packed & kLeafFirstMask);
                    o.count[k] = (packed >> kLeafCountShift) + 1;
                }
            }
        }
    }
    if (sorted_tri_ids && n > 0) CK(cudaMemcpy(sorted_tri_ids, ctx->p_orig, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if ((scene_lo || scene_hi) && n > 0) {
        uint32_t b[12];
        CK(cudaMemcpy(b, ctx->d_bounds.p, sizeof b, cudaMemcpyDeviceToHost));
        auto ord2f = [](uint32_t u) {
            u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
            float f;
            memcpy(&f, &u, 4);
            return f;
        };
        for (int k = 0; k < 3; k++) {
            if (scene_lo) scene_lo[k] = ord2f(b[6 + k]);
            if (scene_hi) scene_hi[k] = ord2f(b[9 + k]);
        }
    }
    return RT_OK;
}

int rt_get_counters(rt_ctx* ctx, rt_counters* out) {
    GUARD();
    if (!out) return fail(ctx, RT_ERR_INVALID, "rt_get_counters: NULL");
    CK(cudaStreamSynchronize(ctx->stream));
    harvest_events(ctx);
    unsigned long long s[4];
    CK(cudaMemcpy(s, ctx->d_stats.p, sizeof s, cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof *out);
    out->segments = s[0];
    out->paths = s[1];
    out->node_visits = s[2];
    out->tri_tests = s[3];
    out->extend_launches = ctx->extend_launches;
    out->kernel_launches = ctx->kernel_launches;
    out->extend_ms = ctx->extend_ms_acc;
    out->shade_ms = ctx->shade_ms_acc;
    out->build_ms = ctx->build_ms;
    out->bvh_nodes = ctx->n_tris >= 2 ? (uint64_t)ctx->n_tris - 1 : 0;
    out->bvh_bytes = out->bvh_nodes * 32 + (uint64_t)ctx->n_tris * 48;
    out->bvh_depth = ctx->bvh_depth;
    out->bvh_width = 2;
    // rendering's k_extend after bounce 0: the counted walk when instrumented, else the one without widening
    out->extend_blocks_per_sm = (uint64_t)ctx->extend_residency.blocks_per_sm[(int)Query::RENDER][ctx->wide_ok][0];
    out->bvh_stack_need = ctx->bvh_depth;
    out->bvh_build_rounds = ctx->build_rounds;
    if (ctx->wide_ok) {  // what k_extend walks: the 4-wide tree
        out->bvh_nodes = ctx->wide_nodes;
        out->bvh_bytes = (uint64_t)ctx->wide_nodes * 64 + (uint64_t)ctx->n_tris * 48;
        out->bvh_depth = (uint64_t)ctx->wide_depth;
        out->bvh_width = 4;
        out->bvh_stack_need = ctx->wide_stack_need;
    }
    return RT_OK;
}

int rt_reset_counters(rt_ctx* ctx) {
    GUARD();
    CK(cudaStreamSynchronize(ctx->stream));
    harvest_events(ctx);
    CK(cudaMemset(ctx->d_stats.p, 0, 4 * sizeof(unsigned long long)));
    ctx->kernel_launches = 0;
    ctx->extend_launches = 0;
    ctx->extend_ms_acc = 0.0;
    ctx->shade_ms_acc = 0.0;
    return RT_OK;
}

int rt_comm_unique_id(uint8_t id_out[128]) {
    if (!id_out) return fail(nullptr, RT_ERR_INVALID, "rt_comm_unique_id: NULL");
    NcclApi& N = nccl();
    if (!N.ok) return fail(nullptr, RT_ERR_NCCL, N.err);
    ncclUniqueId id;
    ncclResult_t r = N.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, RT_ERR_NCCL, "ncclGetUniqueId failed");
    memcpy(id_out, id.internal, 128);
    return RT_OK;
}

int rt_comm_init(rt_ctx* ctx, const uint8_t id[128]) {
    GUARD();
    if (!id) return fail(ctx, RT_ERR_INVALID, "rt_comm_init: NULL id");
    NcclApi& N = nccl();
    if (!N.ok) return fail(ctx, RT_ERR_NCCL, N.err);
    if (ctx->comm) return fail(ctx, RT_ERR_STATE, "rt_comm_init: already initialised");
    ncclUniqueId uid;
    memcpy(uid.internal, id, 128);
    CKN(N.CommInitRank(&ctx->comm, ctx->cfg.world_size, uid, ctx->cfg.rank));
    return RT_OK;
}

int64_t rt_split_rows(int32_t height, int32_t band_rows, int32_t rank, int32_t world, int32_t* rows_out, int64_t cap) {
    if (height <= 0 || world <= 0 || rank < 0 || rank >= world) return 0;
    const int band = band_rows > 0 ? band_rows : 8;
    int64_t n = 0;
    for (int y = 0; y < height; y++) {
        if (((y / band) % world) != rank) continue;
        if (rows_out && n < cap) rows_out[n] = y;
        n++;
    }
    return n;
}

int64_t rt_split_frames(int32_t frames, int32_t rank, int32_t world, int32_t* frames_out, int64_t cap) {
    if (frames <= 0 || world <= 0 || rank < 0 || rank >= world) return 0;
    int64_t n = 0;
    for (int f = 0; f < frames; f++) {
        if ((f % world) != rank) continue;
        if (frames_out && n < cap) frames_out[n] = f;
        n++;
    }
    return n;
}

int rt_plan_batches(uint64_t max_paths_in_flight, int64_t local_pixels, int32_t samples_per_pixel, int32_t frames,
                    int32_t rng_mode, int32_t* samples_per_batch, int32_t* frames_per_batch) {
    if (!samples_per_batch || !frames_per_batch || local_pixels < 0 || samples_per_pixel <= 0 || frames <= 0) return RT_ERR_INVALID;
    int s = 1, f = 1;
    plan_batches(max_paths_in_flight, (size_t)local_pixels, samples_per_pixel, frames, rng_mode == RT_RNG_REF_PCG, &s, &f);
    *samples_per_batch = s;
    *frames_per_batch = f;
    return RT_OK;
}

}  // extern "C"
