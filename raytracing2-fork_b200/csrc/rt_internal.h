// rt_internal.h — declarations shared by the translation units of librt_b200.so (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rt_b200.h"
#include "rt_scene.cuh"

namespace rt {

// ---------------------------------------------------------------- bvh_build.cu
struct BuildArgs {
    const rt_triangle* tris;  // device copy of the caller's array (original order)
    int n;
    int use_ploc;             // 1 = PLOC hierarchy (default), 0 = Karras LBVH
    float4* centroid;         // n
    uint32_t* bounds;         // 12 order-preserving uints
    uint64_t* keys[2];        // n each
    uint32_t* vals[2];        // n each
    uint32_t* hist;           // build_scratch_words(n): sort histograms, later PLOC control block + tile states
    int32_t* children;        // 2*(n-1)
    int32_t* parent;          // 2n-1
    float4* boxes;            // 2*(2n-1)
    uint32_t* flags;          // n+1
    uint32_t* nodeDepth;      // 2n (height of the subtree under each inner node / entity)
    uint32_t* status;         // kBuildStatusWords: depth of the binary tree + error flags (see below)
    int sm_count;
    float* grid;              // 6: quantisation grid (output)
    uint4* nodes;             // 2*(n-1)   (output)
    uint4* nodes4;            // 4*(n-1) or NULL: 4-wide nodes collapsed from the binary tree (output)
    uint32_t* wide_count;     // 2: [0] number of 4-wide nodes written, [1] worst-case traversal stack entries (device)
    int* wide_levels;         // host: depth of the 4-wide tree = levels the collapse ran (output)
    float4* geom;             // 4*n       (output)
    float4* shade;            // 2*n       (output)
    int32_t* orig;            // n         (output)
};
// status words written by the build (device), read back once by rt_scene_build
constexpr int kBuildDepth = 0;       // depth of the binary tree
constexpr int kBuildNonFinite = 1;   // != 0: a vertex coordinate is inf or NaN
constexpr int kBuildPlocStuck = 2;   // != 0: PLOC found no mutual pair / ran out of rounds (caller falls back to Karras)
constexpr int kBuildPlocRounds = 3;  // rounds the clustering took (diagnostic)
constexpr int kBuildStatusWords = 4;
cudaError_t build_lbvh(const BuildArgs& a, cudaStream_t st, uint64_t* launches);
size_t build_scratch_words(int n);
// sets *flag (device word) to 1 if a vertex coordinate is NaN, inf or larger than 1e18 in magnitude
cudaError_t validate_triangles(const rt_triangle* tris, int n, uint32_t* flag, int sm_count, cudaStream_t st);

// ---------------------------------------------------------------- wavefront.cu
// Path state of the wavefront, structure of arrays, 16-byte records, ping-ponged between bounces
// so that every kernel reads and writes dense, coalesced arrays (DESIGN.md §3).
struct PathArrays {
    float4* od0;   // origin.xyz, dir.x
    float4* od1;   // dir.yz, throughput.xy
    float4* misc;  // throughput.z, slot id (bits), rng carry (bits), flags (bits: bounce | insideGlass<<16)
};
// Exact unsigned division by a launch constant (Granlund & Montgomery): q = (t + ((n - t) >> 1)) >> (l - 1) with
// t = umulhi(M, n); valid for every 32-bit n and 2 <= d < 2^31.  d == 1 is flagged by l == 0.
struct FastDiv {
    uint32_t M, l;
};
inline FastDiv make_fastdiv(uint32_t d) {
    FastDiv f{0u, 0u};
    if (d <= 1u) return f;
    uint32_t l = 0;
    while (((uint64_t)1 << l) < d) l++;
    f.M = (uint32_t)((((uint64_t)1 << 32) * (((uint64_t)1 << l) - d)) / d + 1);
    f.l = l;
    return f;
}
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t fastdiv(uint32_t n, FastDiv f) {
    if (f.l == 0u) return n;
    const uint32_t t = __umulhi(f.M, n);
    return (t + ((n - t) >> 1)) >> (f.l - 1u);
}
#endif
struct FrameParams {
    rt_uniforms u;
    int32_t width, height;
    int32_t local_pixels;       // pixels this rank renders
    // One batch of the wavefront holds `lanes_active` lanes of every local pixel; lane L carries sample
    // sample_base + L % samples_in_batch of batch frame L / samples_in_batch, whose frameIndex is
    // u.frameIndex + (L / samples_in_batch) * frame_stride.  Several frames share a batch whenever a whole
    // frame needs fewer path slots than the budget (small images, tile split, RT_RNG_REF_PCG where a pixel's
    // samples are sequential), so the persistent kernels always see large wavefronts.
    int32_t sample_base;        // first sample index of this batch
    int32_t lanes_active;       // frames_in_batch * samples_in_batch
    int32_t frames_in_batch;    // >= 1
    int32_t samples_in_batch;   // samples of one pixel of one frame in flight together (1 in RT_RNG_REF_PCG mode)
    int32_t frame_stride;       // frameIndex step between batch frames (world_size under RT_SPLIT_FRAMES)
    int32_t debug_zero_contrib; // RT_DEBUG_ZERO_CONTRIB=1: raygen clears every contrib slot (debugging aid)
    const int32_t* rows;        // local row -> absolute row (RT_SPLIT_TILES), NULL = identity
    FastDiv div_pixels;         // / local_pixels
    FastDiv div_samples;        // / samples_in_batch
    FastDiv div_width;          // / width
};
struct WaveBuffers {
    PathArrays cur, next;
    float4* hit;          // t, u, v, slot(bits) per path of `cur`
    float4* contrib;      // radiance of each (lane, pixel) slot of the batch
    float4* accum;        // running sum per (batch frame, local pixel) (xyz)
    uint32_t* pix_rng;    // RT_RNG_REF_PCG: the per-(batch frame, pixel) stream state carried across samples
    uint32_t* counts;     // counts[b] = live paths entering bounce b (maxBounce + 2 entries), followed by
                          // the same number of k_extend work cursors
    unsigned long long* stats;  // [0] segments [1] paths [2] node visits [3] tri tests
    float4* image;        // W*H RGBA32F, bottom-up (the reference's image binding 0)
    uint32_t* frame_sum;  // W*H*3 sums of the 8-bit frames, bottom-up
    uint8_t* out_rgb8;    // W*H*3 final, top-down
};

// What k_extend computes.  RENDER: closest hit of every queued path, (t, u, v, sorted slot) into the hit records.
// CLOSEST / ANY (rt_query_closest / rt_query_occluded): the caller's (N, 3) origin and direction arrays are read and
// its outputs written in place, with a per-ray tmax; ANY stops a ray at the first triangle it accepts.  The parity
// hooks (rt_first_hit, rt_trace_rays) are CLOSEST with no tmax on device copies staged by rt_api.cu.
enum class Query : int { RENDER = 0, CLOSEST = 1, ANY = 2 };
// device pointers of one ray query (caller memory, or the hooks' staging; NULL tmax = unbounded, NULL closest outputs =
// skipped)
struct QueryArgs {
    const float* o3;
    const float* d3;
    const float* tmax;
    int32_t* tri;
    float* dst;
    float* bu;
    float* bv;
    uint8_t* occluded;
};

// device pointers of one nearest-triangle query (rt_query_nearest; all caller memory, NULL max_dist = unbounded, NULL
// outputs = skipped)
struct NearestArgs {
    const float* points;    // count * 3
    const float* max_dist;  // count
    int32_t* tri;
    float* dist;
    float* bu;
    float* bv;
    float* closest;         // count * 3
};

// Resident 128-thread blocks per SM of the k_extend instantiation a launch picks, indexed [Q][4-wide][widen] like that
// choice (wavefront.cu, extend_kernel).  Filled once per ctx; a persistent k_extend grid is SMs x this.
struct ExtendResidency {
    int blocks_per_sm[3][2][2];
};

struct Launcher {
    cudaStream_t st;
    int sm_count;
    int rng_mode;
    bool instrument;
    const ExtendResidency* extend_residency;  // of the variants `instrument` selects
    bool widen_primary;  // camera rays may start far outside the quantisation grid (rt_scene.cuh, slab1)
    int shade_blocks_per_sm;  // grid-stride k_shade: blocks per SM
    uint64_t* kernel_launches;
    uint64_t* extend_launches;
    // optional per-class device timing
    cudaEvent_t* ev_pool;
    int ev_cap;
    int* ev_used;
    int* ev_tag;  // 0 extend, 1 other
    bool timing;
};

// fills `r` from the occupancy of each k_extend instantiation a ctx with this `instrument` setting launches
cudaError_t wf_extend_residency(bool instrument, ExtendResidency* r);
cudaError_t wf_clear_accum(const Launcher& L, const WaveBuffers& wb, long long entries);
cudaError_t wf_seed_pixels(const Launcher& L, const SceneView& sc, const WaveBuffers& wb, const FrameParams& fp);
cudaError_t wf_render_batch(const Launcher& L, const SceneView& sc, const WaveBuffers& wb, const FrameParams& fp);
cudaError_t wf_resolve_frame(const Launcher& L, const WaveBuffers& wb, const FrameParams& fp, bool add_to_sum);
cudaError_t wf_preview(const Launcher& L, const SceneView& sc, const WaveBuffers& wb, const FrameParams& fp);
cudaError_t wf_finalize(const Launcher& L, const uint32_t* frame_sum, uint8_t* out, int w, int h, int frames);
// rt_first_hit's width x height camera rays as (N, 3) origin and direction arrays (device)
cudaError_t wf_first_rays(const Launcher& L, const FrameParams& fp, int mode, float* o3, float* d3);
// n > 0 rays of `q` through k_extend (CLOSEST or ANY); counts = [0] rays, [1] work cursor (device words of the ctx)
cudaError_t wf_query(const Launcher& L, const SceneView& sc, const QueryArgs& q, int64_t n, Query mode,
                     uint32_t* counts, unsigned long long* stats);
cudaError_t wf_scatter_rows(const Launcher& L, const uint32_t* compact, uint32_t* full, const int32_t* rows,
                            int nrows, int width);
cudaError_t wf_gather_rows(const Launcher& L, const uint32_t* full, uint32_t* compact, const int32_t* rows,
                           int nrows, int width);

// ---------------------------------------------------------------- nearest.cu
// n > 0 points through k_nearest, one thread per point, on L.st
cudaError_t wf_nearest(const Launcher& L, const SceneView& sc, const NearestArgs& q, int64_t n,
                       unsigned long long* stats);

}  // namespace rt
