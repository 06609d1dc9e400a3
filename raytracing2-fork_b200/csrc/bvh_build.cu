// bvh_build.cu — BVH construction on the GPU (replaces the reference's CPU builder,
// RayTracing/Assets/headers/BVH.h:145-221, called at RayTracing/src/rayTracing.cpp:1293).
//
// Pipeline (all on the ctx stream).  The host reads back 8 bytes at the end of every CHUNK of clustering rounds
// (chunks double: 4, 8, 16, ... rounds) and of every 16 collapse levels — a handful of synchronisations per build
// instead of one per round and per level; everything else, including the cluster counts that size the work,
// stays on the device:
//   k_tri_bounds   per-triangle AABB + centroid, scene centroid bounds by warp shuffle + atomics
//   k_morton       63-bit Morton code of the centroid (21 bits / axis)
//   radix sort     hand-written stable LSD sort of (code, index): 8 passes x 8 bits, each pass
//                  = histogram (k_hist) -> exclusive scan over [digit][block] (k_scan) -> stable
//                  scatter with warp match-any ranking (k_scatter)
//   hierarchy, one of
//     PLOC (default): parallel locally-ordered clustering (Meister & Bittner 2018) over the Morton
//                  order: every round each cluster finds the neighbour within +-kPlocRadius that
//                  minimises the surface area of the union (k_ploc_nn), mutual pairs merge and survivors are
//                  compacted in ONE kernel (k_ploc_merge_scan: flags, single-pass decoupled-look-back prefix
//                  scan over all tiles, merge); once <= 2048 clusters remain a single block finishes every
//                  remaining round in shared memory (k_ploc_tail) — that is where the long chains are.  An offline
//                  comparison (tools/bvh_quality.cpp) on the config-2 scene: 20.2 node visits per
//                  diffuse ray against 31.0 for the Karras tree — traversal cost is what the
//                  benchmark measures, the build stays ~2 ms.
//     Karras     : k_hierarchy (one thread per inner node finds its range and split) + k_refit
//                  (bottom-up AABB union with one atomic flag per inner node); RT_BVH_BUILDER=lbvh
//   k_emit_nodes   32-byte nodes: both child boxes in the parent, 16-bit planes rounded outward
//   k_emit_tris    sorted triangle records: (a, e0, e1, N, unit normal, material) | (uvs, material, orig)
// Everything is deterministic (stable sort, min/max are order independent), so every GPU of a
// multi-GPU job builds the identical tree.
#include <cstdio>
#include <cstdlib>

#include "rt_internal.h"

namespace rt {

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f2ord(float f) {  // order-preserving float → uint
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// bounds[0..2] = min of centroids, [3..5] = max of centroids, [6..8] = scene min, [9..11] = scene max
// (order-preserving uints)
__global__ void k_init_bounds(uint32_t* bounds) {
    const int i = threadIdx.x;
    if (i < 12) bounds[i] = ((i % 6) < 3) ? 0xffffffffu : 0u;
}

__global__ void __launch_bounds__(256) k_tri_bounds(const rt_triangle* __restrict__ tris, int n,
                                                    float4* __restrict__ centroid,
                                                    uint32_t* __restrict__ bounds, uint32_t* __restrict__ status) {
    bool bad = false;
    float cmin[3] = {3.4e38f, 3.4e38f, 3.4e38f}, cmax[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    float smin[3] = {3.4e38f, 3.4e38f, 3.4e38f}, smax[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 a = *reinterpret_cast<const float4*>(tris[i].a);
        const float4 b = *reinterpret_cast<const float4*>(tris[i].b);
        const float4 c = *reinterpret_cast<const float4*>(tris[i].c);
        const float lo[3] = {fminf(fminf(a.x, b.x), c.x), fminf(fminf(a.y, b.y), c.y), fminf(fminf(a.z, b.z), c.z)};
        const float hi[3] = {fmaxf(fmaxf(a.x, b.x), c.x), fmaxf(fmaxf(a.y, b.y), c.y), fmaxf(fmaxf(a.z, b.z), c.z)};
        float ce[3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            ce[k] = 0.5f * lo[k] + 0.5f * hi[k];
            cmin[k] = fminf(cmin[k], ce[k]);
            cmax[k] = fmaxf(cmax[k], ce[k]);
            smin[k] = fminf(smin[k], lo[k]);
            smax[k] = fmaxf(smax[k], hi[k]);
        }
        centroid[i] = make_float4(ce[0], ce[1], ce[2], 0.0f);
        // inf - inf and NaN both fail this test; such a triangle has no box to cluster by
        bad |= !(hi[0] - lo[0] < 3.0e38f && hi[1] - lo[1] < 3.0e38f && hi[2] - lo[2] < 3.0e38f);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(&status[kBuildNonFinite], 1u);
#pragma unroll
    for (int k = 0; k < 3; k++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            cmin[k] = fminf(cmin[k], __shfl_xor_sync(0xffffffffu, cmin[k], off));
            cmax[k] = fmaxf(cmax[k], __shfl_xor_sync(0xffffffffu, cmax[k], off));
            smin[k] = fminf(smin[k], __shfl_xor_sync(0xffffffffu, smin[k], off));
            smax[k] = fmaxf(smax[k], __shfl_xor_sync(0xffffffffu, smax[k], off));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            atomicMin(&bounds[k], f2ord(cmin[k]));
            atomicMax(&bounds[3 + k], f2ord(cmax[k]));
            atomicMin(&bounds[6 + k], f2ord(smin[k]));
            atomicMax(&bounds[9 + k], f2ord(smax[k]));
        }
    }
}

// Upload-time validation (rt_scene_set_triangles): a vertex coordinate that is NaN, inf or beyond 1e18 in magnitude.
// Within that range every box extent and every surface area the builder forms stays finite, so the build itself can
// run without ever looking at a status word on the host.  One pass at HBM speed, read back with the sync the upload
// needs anyway.
__global__ void __launch_bounds__(256) k_validate_tris(const rt_triangle* __restrict__ tris, int n,
                                                       uint32_t* __restrict__ flag) {
    bool bad = false;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 a = *reinterpret_cast<const float4*>(tris[i].a);
        const float4 b = *reinterpret_cast<const float4*>(tris[i].b);
        const float4 c = *reinterpret_cast<const float4*>(tris[i].c);
        const float m = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(b.x))),
                              fmaxf(fmaxf(fabsf(b.y), fabsf(b.z)), fmaxf(fabsf(c.x), fmaxf(fabsf(c.y), fabsf(c.z)))));
        // fmaxf drops NaN operands, so test them separately: x != x
        const bool nan = a.x != a.x || a.y != a.y || a.z != a.z || b.x != b.x || b.y != b.y || b.z != b.z ||
                         c.x != c.x || c.y != c.y || c.z != c.z;
        bad |= nan || !(m <= 1.0e18f);
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}
cudaError_t validate_triangles(const rt_triangle* tris, int n, uint32_t* flag, int sm_count, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(flag, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess || n <= 0) return e;
    const int blocks = std::min((n + 255) / 256, sm_count * 8);
    k_validate_tris<<<blocks, 256, 0, st>>>(tris, n, flag);
    return cudaGetLastError();
}

__device__ __forceinline__ uint64_t spread21(uint32_t v) {  // 21 bits → every third bit
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void __launch_bounds__(256) k_morton(const float4* __restrict__ centroid, int n,
                                                const uint32_t* __restrict__ bounds,
                                                uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 c = centroid[i];
    const float cc[3] = {c.x, c.y, c.z};
    uint32_t q[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const float lo = ord2f(bounds[k]), hi = ord2f(bounds[3 + k]);
        const float ext = hi - lo;
        float t = ext > 0.0f ? (cc[k] - lo) / ext : 0.0f;
        t = fminf(fmaxf(t, 0.0f), 1.0f);
        q[k] = min((uint32_t)(t * 2097152.0f), 2097151u);
    }
    keys[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    vals[i] = (uint32_t)i;
}

// --------------------------------------------------------------------------------------------- radix sort
constexpr int kSortThreads = 256;
constexpr int kSortItems = 8;                                // keys per thread
constexpr int kSortTile = kSortThreads * kSortItems;         // 2048 keys per block
constexpr int kSortWarps = kSortThreads / 32;

__global__ void __launch_bounds__(kSortThreads) k_hist(const uint64_t* __restrict__ keys, int n, int shift,
                                                       uint32_t* __restrict__ hist, int nblocks) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * kSortTile;
#pragma unroll
    for (int k = 0; k < kSortItems; k++) {
        const int i = base + k * kSortThreads + threadIdx.x;
        if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];  // digit-major
}

// exclusive scan of the digit-major histogram (256 * nblocks entries) by a single block: enough for
// ~10^7 keys (nblocks ~ 5000 → 1.3 M entries, <100 us), and it keeps the pass deterministic.
__global__ void __launch_bounds__(1024) k_scan(uint32_t* __restrict__ hist, int total) {
    __shared__ uint32_t warpSums[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < total; base += 1024 * 4) {
        const int i0 = base + threadIdx.x * 4;
        uint32_t v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = (i0 + k < total) ? hist[i0 + k] : 0u;
        const uint32_t mine = v[0] + v[1] + v[2] + v[3];
        uint32_t incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, off);
            if ((threadIdx.x & 31) >= off) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warpSums[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = warpSums[threadIdx.x];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, w, off);
                if (threadIdx.x >= off) w += t;
            }
            warpSums[threadIdx.x] = w;
        }
        __syncthreads();
        const uint32_t warpBase = (threadIdx.x >> 5) ? warpSums[(threadIdx.x >> 5) - 1] : 0u;
        uint32_t run = carry + warpBase + incl - mine;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (i0 + k < total) hist[i0 + k] = run;
            run += v[k];
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = run;
        __syncthreads();
    }
    if (threadIdx.x == 0) hist[total] = carry;  // grand total in the slot after the last element
}

// Stable scatter.  Key order inside a block is (warp, item, lane): warp w owns the contiguous strip
// [w*256, (w+1)*256) of the tile and walks it 32 keys at a time, so ranking by (earlier warps,
// earlier items of my warp, lower lanes) preserves the input order of equal digits.
__global__ void __launch_bounds__(kSortThreads) k_scatter(const uint64_t* __restrict__ keysIn,
                                                          const uint32_t* __restrict__ valsIn,
                                                          uint64_t* __restrict__ keysOut,
                                                          uint32_t* __restrict__ valsOut, int n, int shift,
                                                          const uint32_t* __restrict__ hist, int nblocks) {
    __shared__ uint32_t warpCount[kSortWarps][256];
    __shared__ uint32_t digitBase[256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int d = lane; d < 256; d += 32) warpCount[warp][d] = 0;
    digitBase[threadIdx.x] = hist[threadIdx.x * nblocks + blockIdx.x];
    __syncwarp();

    const int stripBase = blockIdx.x * kSortTile + warp * (32 * kSortItems);
    uint64_t key[kSortItems];
    uint32_t rank[kSortItems];
#pragma unroll
    for (int k = 0; k < kSortItems; k++) {
        const int i = stripBase + k * 32 + lane;
        const bool valid = i < n;
        key[k] = valid ? keysIn[i] : ~0ull;
        const uint32_t digit = (uint32_t)(key[k] >> shift) & 255u;
        // invalid lanes vote in a private group so they never disturb real digits
        const uint32_t peers = __match_any_sync(0xffffffffu, valid ? digit : 256u + lane);
        const uint32_t below = __popc(peers & ((1u << lane) - 1u));
        uint32_t base = 0;
        if (valid) {
            const int leader = __ffs(peers) - 1;
            if (lane == leader) {
                base = warpCount[warp][digit];
                warpCount[warp][digit] = base + __popc(peers);
            }
            base = __shfl_sync(peers, base, leader);
        }
        rank[k] = base + below;
        __syncwarp();
    }
    __syncthreads();
    // exclusive prefix over warps, per digit (thread d handles digit d)
    {
        uint32_t run = digitBase[threadIdx.x];
#pragma unroll
        for (int w = 0; w < kSortWarps; w++) {
            const uint32_t c = warpCount[w][threadIdx.x];
            warpCount[w][threadIdx.x] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kSortItems; k++) {
        const int i = stripBase + k * 32 + lane;
        if (i < n) {
            const uint32_t digit = (uint32_t)(key[k] >> shift) & 255u;
            const uint32_t pos = warpCount[warp][digit] + rank[k];
            keysOut[pos] = key[k];
            valsOut[pos] = valsIn[i];
        }
    }
}

// The histogram kernel must bin keys with the same (warp, item, lane) → block mapping only at block
// granularity, which it does: both kernels give block b the keys [b*2048, (b+1)*2048).

// --------------------------------------------------------------------------------------------- Karras
__device__ __forceinline__ int delta(const uint64_t* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const uint64_t a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz((uint32_t)i ^ (uint32_t)j);
    return __clzll((long long)(a ^ b));
}

// children[2*i], children[2*i+1]: >= 0 inner node, < 0 leaf ~slot.  parent[node] for inner nodes,
// parent[n-1+slot] for leaves.
__global__ void __launch_bounds__(256) k_hierarchy(const uint64_t* __restrict__ keys, int n,
                                                   int32_t* __restrict__ children,
                                                   int32_t* __restrict__ parent) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(keys, n, i, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int32_t left = (lo == gamma) ? ~gamma : gamma;
    const int32_t right = (hi == gamma + 1) ? ~(gamma + 1) : (gamma + 1);
    children[2 * i] = left;
    children[2 * i + 1] = right;
    if (left >= 0) parent[left] = i; else parent[n - 1 + gamma] = i;
    if (right >= 0) parent[right] = i; else parent[n - 1 + gamma + 1] = i;
    if (i == 0) parent[0] = -1;
}

// boxes: 2 float4 per entity (lo, hi); entities 0..n-2 inner nodes, n-1.. leaves (by sorted slot)
__global__ void __launch_bounds__(256) k_refit(const rt_triangle* __restrict__ tris,
                                               const uint32_t* __restrict__ sortedIdx, int n,
                                               const uint32_t* __restrict__ bounds,
                                               const int32_t* __restrict__ children,
                                               const int32_t* __restrict__ parent,
                                               float4* __restrict__ boxes, uint32_t* __restrict__ flags,
                                               uint32_t* __restrict__ nodeDepth, uint32_t* __restrict__ maxDepth) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const rt_triangle& t = tris[sortedIdx[s]];
    // Leaf boxes are padded like the reference's (BVH.h:47-51, 1e-4) and by 2e-6 of the scene extent:
    // the exact triangle test and the slab test round differently, the pad keeps every accepted hit
    // strictly inside its leaf's slabs.
    float ext = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; k++) ext = fmaxf(ext, ord2f(bounds[9 + k]) - ord2f(bounds[6 + k]));
    const float pad = fmaxf(1e-4f, 2e-6f * ext);
    float lo[3], hi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = fminf(fminf(t.a[k], t.b[k]), t.c[k]) - pad;
        hi[k] = fmaxf(fmaxf(t.a[k], t.b[k]), t.c[k]) + pad;
    }
    boxes[2 * (n - 1 + s)] = make_float4(lo[0], lo[1], lo[2], 0.0f);
    boxes[2 * (n - 1 + s) + 1] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    if (n == 1) return;
    __threadfence();
    int node = parent[n - 1 + s];
    uint32_t depth = 1;
    while (node >= 0) {
        // both arrivals deposit the height of their subtree; the second one continues with the max
        atomicMax(&nodeDepth[node], depth);
        __threadfence();
        if (atomicAdd(&flags[node], 1u) == 0u) return;  // first arrival: the sibling is not ready yet
        __threadfence();
        depth = __ldcg(&nodeDepth[node]);
        const int32_t cl = children[2 * node], cr = children[2 * node + 1];
        const int el = cl >= 0 ? cl : (n - 1 + ~cl), er = cr >= 0 ? cr : (n - 1 + ~cr);
        // the sibling's box was written by another SM: read through L2, never a stale L1 line
        const float4 llo = __ldcg(&boxes[2 * el]);
        const float4 lhi = __ldcg(&boxes[2 * el + 1]);
        const float4 rlo = __ldcg(&boxes[2 * er]);
        const float4 rhi = __ldcg(&boxes[2 * er + 1]);
        boxes[2 * node] = make_float4(fminf(llo.x, rlo.x), fminf(llo.y, rlo.y), fminf(llo.z, rlo.z), 0.0f);
        boxes[2 * node + 1] = make_float4(fmaxf(lhi.x, rhi.x), fmaxf(lhi.y, rhi.y), fmaxf(lhi.z, rhi.z), 0.0f);
        __threadfence();
        node = parent[node];
        depth++;
    }
    atomicMax(maxDepth, depth);
}

// --------------------------------------------------------------------------------------------- PLOC
// search window of the clustering.  Measured on config 2 (profiles/r2_knobs_ab.txt):
// radius 6 -> 7.13 wide-node visits per segment, 10 -> 7.24, 16 / 25 / 40 -> slightly MORE visits and a slower build.
constexpr int kPlocRadiusDefault = 6;

// leaf boxes in Morton order (entity n-1+slot), cluster list = all leaves
__global__ void __launch_bounds__(256) k_ploc_init(const rt_triangle* __restrict__ tris,
                                                   const uint32_t* __restrict__ sortedIdx, int n,
                                                   const uint32_t* __restrict__ bounds, float4* __restrict__ boxes,
                                                   int32_t* __restrict__ cluster, uint32_t* __restrict__ height) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const rt_triangle& t = tris[sortedIdx[s]];
    float ext = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; k++) ext = fmaxf(ext, ord2f(bounds[9 + k]) - ord2f(bounds[6 + k]));
    const float pad = fmaxf(1e-4f, 2e-6f * ext);  // same padding rule as k_refit
    float lo[3], hi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = fminf(fminf(t.a[k], t.b[k]), t.c[k]) - pad;
        hi[k] = fmaxf(fmaxf(t.a[k], t.b[k]), t.c[k]) + pad;
    }
    // .w of the lower corner = SAH cost of the subtree given that its box is hit (one triangle test = 1),
    // .w of the upper corner = triangles it holds AS A LEAF (0 = inner node that stays split)
    boxes[2 * (n - 1 + s)] = make_float4(lo[0], lo[1], lo[2], 1.0f);
    boxes[2 * (n - 1 + s) + 1] = make_float4(hi[0], hi[1], hi[2], __int_as_float(1));
    cluster[s] = ~s;
    height[n - 1 + s] = 0u;
}

__device__ __forceinline__ int entity_of(int32_t c, int n) { return c >= 0 ? c : (n - 1 + ~c); }
__device__ __forceinline__ float union_area(float4 alo, float4 ahi, float4 blo, float4 bhi) {
    const float dx = fmaxf(ahi.x, bhi.x) - fminf(alo.x, blo.x);
    const float dy = fmaxf(ahi.y, bhi.y) - fminf(alo.y, blo.y);
    const float dz = fmaxf(ahi.z, bhi.z) - fminf(alo.z, blo.z);
    return dx * dy + dy * dz + dz * dx;  // symmetric in a,b bit for bit
}

// ---- device-side control of the clustering rounds ------------------------------------------------------------
// ctl (uint32 words in the dead sort-histogram buffer), double buffered by round parity so that a round can read
// its cluster count while its last tile publishes the next one:
//   ctl[4 * (round & 1) + 0] = m        clusters entering the round
//   ctl[4 * (round & 1) + 1] = created  inner nodes created so far
//   ctl[4 * (round & 1) + 2] = buf      which of the two cluster lists is current (a round that has nothing to
//                                       do — the count is already small enough for the tail — moves no data)
//   ctl[8]                   = ticket   tile ids of the look-back scan are handed out in arrival order
// tileState[t] (uint64): bits 63..62 = 0 invalid / 1 tile aggregate / 2 inclusive prefix; bits 59..32 = kept
// clusters, bits 31..0 = merged pairs.
constexpr int kPlocTile = 1024;        // clusters per tile of the scan (256 threads x 4)
constexpr int kPlocTailMax = 2048;     // clusters a single block finishes on its own
constexpr int kCtlTicket = 8;
constexpr int kCtlWords = 16;
constexpr unsigned long long kTileAgg = 1ull << 62, kTileIncl = 2ull << 62, kTileFlagMask = 3ull << 62;

// (no __restrict__ here: k_ploc_tail reads boxes that the same kernel wrote in its previous round)
__device__ __forceinline__ int ploc_nearest(const int32_t* cluster, int i, int m, int n, const float4* boxes, int radius) {
    const int ei = entity_of(cluster[i], n);
    const float4 lo = boxes[2 * ei], hi = boxes[2 * ei + 1];
    float best = 3.4e38f;
    int bj = -1;
    const int j0 = max(0, i - radius), j1 = min(m - 1, i + radius);
    for (int j = j0; j <= j1; j++) {
        if (j == i) continue;
        const int ej = entity_of(cluster[j], n);
        const float a = union_area(lo, hi, boxes[2 * ej], boxes[2 * ej + 1]);
        // Ties go to the lowest position: the globally smallest pair is then always mutual, so every
        // round merges at least one pair.  (A symmetric i^j tie-break pairs up runs of identical boxes in
        // one round, but on regular meshes it also changes which of many equal-area candidates merge and
        // measured 4 % slower traversal on config 2 through a worse node layout; runs of exact duplicates
        // just take more rounds.)
        if (a < best) {
            best = a;
            bj = j;
        }
    }
    return bj;
}

// Leaves of more than one triangle.  The two triangles of a quad have almost the same box, so a tree with one
// triangle per leaf makes every ray that touches the quad test two boxes, push and pop one of them, and visit two
// leaves (ncu, round 2: the leaf phase of k_extend was 22 % of its warp instructions at ~9 active lanes, 4.25
// triangle tests per segment).  At every merge the builder compares, bottom-up, the SAH cost of keeping the node
// split, 2 Cb + (A_a cost_a + A_b cost_b) / A, with the cost of one leaf holding all its triangles, count x 1, and
// marks the node as a leaf when that is cheaper and the count allowed.  Cb = cost of a box test relative to a
// triangle test, maxTris = 1 switches the feature off.
struct LeafPolicy {
    float cb;
    int maxTris;
};
__device__ __forceinline__ float box_area(float4 lo, float4 hi) {
    const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}
// one merge: node `id` = union of clusters a and b
__device__ __forceinline__ void ploc_make_node(int id, int32_t a, int32_t b, int n, float4* __restrict__ boxes,
                                               int32_t* __restrict__ children, uint32_t* __restrict__ height,
                                               int32_t* __restrict__ parentOf, uint32_t* __restrict__ innerCount,
                                               int32_t* __restrict__ leafParent, LeafPolicy pol) {
    const int ea = entity_of(a, n), eb = entity_of(b, n);
    const float4 alo = boxes[2 * ea], ahi = boxes[2 * ea + 1], blo = boxes[2 * eb], bhi = boxes[2 * eb + 1];
    float4 lo = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.0f);
    float4 hi = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.0f);
    const int la = __float_as_int(ahi.w), lb = __float_as_int(bhi.w);
    const float area = box_area(lo, hi);
    const float split = 2.0f * pol.cb + (area > 0.0f ? (box_area(alo, ahi) * alo.w + box_area(blo, bhi) * blo.w) / area
                                                     : alo.w + blo.w);
    const float leaf = (float)(la + lb);
    // the root (id 0, the last node created) always stays an inner node: the traversal starts at an inner node
    const bool asLeaf = id != 0 && la > 0 && lb > 0 && la + lb <= pol.maxTris && leaf <= split;
    lo.w = asLeaf ? leaf : split;
    hi.w = __int_as_float(asLeaf ? la + lb : 0);
    boxes[2 * id] = lo;
    boxes[2 * id + 1] = hi;
    children[2 * id] = a;
    children[2 * id + 1] = b;
    height[id] = max(height[ea], height[eb]) + 1u;
    // bookkeeping for the depth-first relabelling: parent links and inner nodes per subtree
    if (a >= 0) parentOf[a] = id; else leafParent[~a] = id;
    if (b >= 0) parentOf[b] = id; else leafParent[~b] = id;
    innerCount[id] = 1u + (a >= 0 ? innerCount[a] : 0u) + (b >= 0 ? innerCount[b] : 0u);
}

__global__ void k_ploc_ctl_init(uint32_t* __restrict__ ctl, int n) {
    if (threadIdx.x < kCtlWords) ctl[threadIdx.x] = 0u;
    __syncwarp();
    if (threadIdx.x == 0) ctl[0] = (uint32_t)n;
}

// nearest neighbour in the window; also re-arms the scan of this round (ticket, tile states)
__global__ void __launch_bounds__(256) k_ploc_nn(int n, int round, uint32_t* __restrict__ ctl,
                                                 unsigned long long* __restrict__ tileState,
                                                 const int32_t* __restrict__ cluster0,
                                                 const int32_t* __restrict__ cluster1,
                                                 const float4* __restrict__ boxes, int32_t* __restrict__ nn, int radius) {
    const uint32_t* cin = ctl + 4 * (round & 1);
    uint32_t* cout = ctl + 4 * ((round + 1) & 1);
    const int m = (int)cin[0];
    const int32_t* cluster = cin[2] ? cluster1 : cluster0;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        ctl[kCtlTicket] = 0u;
        if (m <= kPlocTailMax) {  // nothing (more) to do globally: the round is a no-op, the state moves on unchanged
            cout[0] = cin[0];
            cout[1] = cin[1];
            cout[2] = cin[2];
        }
    }
    if (m <= kPlocTailMax) return;
    if (i < (m + kPlocTile - 1) / kPlocTile) tileState[i] = 0ull;
    if (i >= m) return;
    nn[i] = ploc_nearest(cluster, i, m, n, boxes, radius);
}

// Flags (mutual pair -> the lower position creates a node, the upper one disappears), exclusive prefix sums of
// "kept" and "merged" over ALL clusters in a single pass (decoupled look-back over the tiles, Merrill & Garland),
// and the merge itself.  The last tile publishes the next round's cluster count.
__global__ void __launch_bounds__(256) k_ploc_merge_scan(int n, int round, uint32_t* __restrict__ ctl,
                                                         unsigned long long* __restrict__ tileState,
                                                         int32_t* __restrict__ cluster0, int32_t* __restrict__ cluster1,
                                                         const int32_t* __restrict__ nn, float4* __restrict__ boxes,
                                                         int32_t* __restrict__ children, uint32_t* __restrict__ height,
                                                         int32_t* __restrict__ parentOf,
                                                         uint32_t* __restrict__ innerCount,
                                                         int32_t* __restrict__ leafParent, LeafPolicy pol,
                                                         uint32_t* __restrict__ status) {
    const uint32_t* cin = ctl + 4 * (round & 1);
    uint32_t* cout = ctl + 4 * ((round + 1) & 1);
    const int m = (int)cin[0];
    const int created = (int)cin[1];
    const uint32_t buf = cin[2];
    const int32_t* clusterIn = buf ? cluster1 : cluster0;
    int32_t* clusterOut = buf ? cluster0 : cluster1;
    if (m <= kPlocTailMax) return;
    __shared__ uint32_t sTile;
    __shared__ unsigned long long sWarp[8];
    __shared__ unsigned long long sPrefix;
    if (threadIdx.x == 0) sTile = atomicAdd(&ctl[kCtlTicket], 1u);
    __syncthreads();
    const int tile = (int)sTile;
    const int tiles = (m + kPlocTile - 1) / kPlocTile;
    if (tile >= tiles) return;

    const int base = tile * kPlocTile + threadIdx.x * 4;
    int32_t c[4];
    int j[4];
    bool mutual[4];
    unsigned long long mine = 0ull;  // kept << 32 | merged
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int i = base + k;
        j[k] = -1;
        mutual[k] = false;
        c[k] = 0;
        if (i < m) {
            j[k] = nn[i];
            mutual[k] = j[k] >= 0 && nn[j[k]] == i;
            c[k] = clusterIn[i];
            const bool keep = !mutual[k] || i < j[k];
            const bool merge = mutual[k] && i < j[k];
            mine += ((unsigned long long)(keep ? 1u : 0u) << 32) | (unsigned long long)(merge ? 1u : 0u);
        }
    }
    // block-wide inclusive scan of the per-thread sums
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
    }
    if (lane == 31) sWarp[warp] = incl;
    __syncthreads();
    unsigned long long warpBase = 0ull, tileTotal = 0ull;
#pragma unroll
    for (int w = 0; w < 8; w++) {
        if (w < warp) warpBase += sWarp[w];
        tileTotal += sWarp[w];
    }
    // look-back: thread 0 publishes the tile aggregate, then sums its predecessors until one holds an inclusive prefix
    if (threadIdx.x == 0) {
        volatile unsigned long long* ts = tileState;
        unsigned long long prefix = 0ull;
        if (tile == 0) {
            ts[0] = kTileIncl | tileTotal;
        } else {
            ts[tile] = kTileAgg | tileTotal;
            __threadfence();
            for (int t = tile - 1; t >= 0; t--) {
                unsigned long long v;
                do { v = ts[t]; } while ((v & kTileFlagMask) == 0ull);
                prefix += v & ~kTileFlagMask;
                if ((v & kTileFlagMask) == kTileIncl) break;
            }
            ts[tile] = kTileIncl | (prefix + tileTotal);
        }
        __threadfence();
        sPrefix = prefix;
        if (tile == tiles - 1) {  // grand totals: the state of the next round
            const unsigned long long total = prefix + tileTotal;
            const uint32_t kept = (uint32_t)(total >> 32), merged = (uint32_t)(total & 0xffffffffu);
            if (merged == 0u) {  // no mutual pair (union areas overflowed): give up, the caller builds a Karras tree
                status[kBuildPlocStuck] = 1u;
                cout[0] = 0u;
            } else {
                cout[0] = kept;
            }
            cout[1] = (uint32_t)created + merged;
            cout[2] = buf ^ 1u;
            status[kBuildPlocRounds] = (uint32_t)round + 1u;
        }
    }
    __syncthreads();
    unsigned long long run = sPrefix + warpBase + incl - mine;  // exclusive prefix of this thread's first item
    const int firstId = (n - 2) - created;  // node ids are handed out from the top: the last node created (the root) is 0
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int i = base + k;
        if (i >= m) break;
        const bool upper = mutual[k] && i > j[k];
        if (!upper) {
            int32_t out = c[k];
            if (mutual[k]) {
                const int id = firstId - (int)(uint32_t)(run & 0xffffffffu);
                ploc_make_node(id, c[k], clusterIn[j[k]], n, boxes, children, height, parentOf, innerCount, leafParent, pol);
                out = id;
                run += 1ull;
            }
            clusterOut[(uint32_t)(run >> 32)] = out;
            run += 1ull << 32;
        }
    }
}

// The last <= kPlocTailMax clusters: one block runs every remaining round (nearest neighbour, flags, scan, merge)
// with the cluster list in shared memory.  Most ROUNDS of a build happen here — the cluster count falls
// geometrically at first and then the large clusters absorb the stragglers one or two per round.
__global__ void __launch_bounds__(1024) k_ploc_tail(int n, int round, uint32_t* __restrict__ ctl,
                                                    const int32_t* __restrict__ cluster0,
                                                    const int32_t* __restrict__ cluster1, float4* __restrict__ boxes,
                                                    int32_t* __restrict__ children, uint32_t* __restrict__ height,
                                                    int32_t* __restrict__ parentOf, uint32_t* __restrict__ innerCount,
                                                    int32_t* __restrict__ leafParent, LeafPolicy pol,
                                                    uint32_t* __restrict__ status, int radius) {
    uint32_t* cio = ctl + 4 * (round & 1);
    int m = (int)cio[0];
    int created = (int)cio[1];
    const int32_t* clusterIn = cio[2] ? cluster1 : cluster0;
    if (m <= 1 || m > kPlocTailMax) return;
    __shared__ int32_t cl[2][kPlocTailMax];
    __shared__ int32_t snn[kPlocTailMax];
    __shared__ uint32_t sWarp[32];
    __shared__ uint32_t sTotal;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int i = t; i < m; i += 1024) cl[0][i] = clusterIn[i];
    __syncthreads();
    int cur = 0;
    uint32_t rounds = (uint32_t)round;
    bool stuck = false;
    while (m > 1) {
        for (int i = t; i < m; i += 1024) snn[i] = ploc_nearest(cl[cur], i, m, n, boxes, radius);
        __syncthreads();
        // items 2t, 2t+1; packed sums: kept << 16 | merged (both <= 2048)
        uint32_t mine = 0u;
        bool mutual[2];
        int j[2];
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int i = 2 * t + k;
            j[k] = -1;
            mutual[k] = false;
            if (i < m) {
                j[k] = snn[i];
                mutual[k] = j[k] >= 0 && snn[j[k]] == i;
                mine += ((!mutual[k] || i < j[k]) ? (1u << 16) : 0u) | ((mutual[k] && i < j[k]) ? 1u : 0u);
            }
        }
        uint32_t incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += v;
        }
        if (lane == 31) sWarp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = sWarp[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, w, off);
                if (lane >= off) w += v;
            }
            sWarp[lane] = w;  // inclusive over warps
            if (lane == 31) sTotal = w;
        }
        __syncthreads();
        uint32_t run = (warp ? sWarp[warp - 1] : 0u) + incl - mine;
        const uint32_t total = sTotal;
        const int firstId = (n - 2) - created;
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int i = 2 * t + k;
            if (i >= m) break;
            const bool upper = mutual[k] && i > j[k];
            if (!upper) {
                int32_t out = cl[cur][i];
                if (mutual[k]) {
                    const int id = firstId - (int)(run & 0xffffu);
                    ploc_make_node(id, out, cl[cur][j[k]], n, boxes, children, height, parentOf, innerCount, leafParent, pol);
                    out = id;
                    run += 1u;
                }
                cl[cur ^ 1][run >> 16] = out;
                run += 1u << 16;
            }
        }
        rounds++;
        const uint32_t merged = total & 0xffffu;
        if (merged == 0u) { stuck = true; break; }
        created += (int)merged;
        m = (int)(total >> 16);
        cur ^= 1;
        __syncthreads();  // node boxes / heights written above are read by everybody in the next round
    }
    if (t == 0) {
        cio[0] = stuck ? 0u : 1u;
        cio[1] = (uint32_t)created;
        status[kBuildPlocRounds] = rounds;
        if (stuck) status[kBuildPlocStuck] = 1u;
    }
}

// Depth-first (pre-order) position of every inner node: walk up to the root adding 1 per level and
// the size of the left sibling's subtree whenever the node is a right child.  A left child then sits
// right behind its parent — in the same 128-byte line three times out of four — and every subtree is
// contiguous in memory.
__global__ void __launch_bounds__(256) k_dfs_order(int n, const int32_t* __restrict__ children,
                                                   const int32_t* __restrict__ parentOf,
                                                   const uint32_t* __restrict__ innerCount, int32_t* __restrict__ order,
                                                   int32_t* __restrict__ firstTri) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    uint32_t pos = 0, tris = 0;
    int node = i;
    while (node != 0) {
        const int p = parentOf[node];
        const int32_t left = children[2 * p];
        pos += 1u;
        if (left != node) {  // we hang on the right: the whole left sibling comes first
            if (left >= 0) pos += innerCount[left];
            tris += left >= 0 ? innerCount[left] + 1u : 1u;  // a binary subtree has one leaf more than inner nodes
        }
        node = p;
    }
    order[i] = (int32_t)pos;
    firstTri[i] = (int32_t)tris;  // triangles stored in front of this subtree's
}
// The same walk from every triangle: its place in the depth-first order of the leaves.  Triangle records are stored
// in this order, so that the triangles of any subtree — in particular of a multi-triangle leaf — are contiguous.
__global__ void __launch_bounds__(256) k_tri_order(int n, const int32_t* __restrict__ children,
                                                   const int32_t* __restrict__ parentOf,
                                                   const int32_t* __restrict__ leafParent,
                                                   const uint32_t* __restrict__ innerCount, int32_t* __restrict__ triPos) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t tris = 0;
    int32_t me = ~s;
    int p = leafParent[s];
    for (;;) {
        const int32_t left = children[2 * p];
        if (left != me) tris += left >= 0 ? innerCount[left] + 1u : 1u;
        if (p == 0) break;
        me = p;
        p = parentOf[p];
    }
    triPos[s] = (int32_t)tris;
}

__global__ void k_ploc_depth(const uint32_t* __restrict__ height, uint32_t* __restrict__ maxDepth) {
    if (threadIdx.x == 0) *maxDepth = height[0] + 1u;
}

// Grid of the quantised boxes: 65535 cells over the scene box padded by 2 leaf pads per side.
// grid[0..2] = world position of coordinate 0, grid[3..5] = cells per world unit.
__global__ void k_grid(const uint32_t* __restrict__ bounds, float* __restrict__ grid) {
    const int k = threadIdx.x;
    if (k >= 3) return;
    float ext = 0.0f;
    for (int a = 0; a < 3; a++) ext = fmaxf(ext, ord2f(bounds[9 + a]) - ord2f(bounds[6 + a]));
    const float pad = 2.0f * fmaxf(1e-4f, 2e-6f * ext);
    const float lo = ord2f(bounds[6 + k]) - pad, hi = ord2f(bounds[9 + k]) + pad;
    grid[k] = lo;
    grid[3 + k] = 65535.0f / fmaxf(hi - lo, 1e-30f);
}

// How a child of the build tree appears in the emitted nodes: a triangle (c < 0) or an inner node marked as a leaf
// becomes a packed leaf reference (first triangle record, count); any other inner node is returned as is (>= 0).
// triPos / firstTri are NULL for the Karras tree: one triangle per leaf, records in Morton order.
struct LeafView {
    const float4* boxes;
    const int32_t* triPos;
    const int32_t* firstTri;
    int n;
    __device__ __forceinline__ bool is_leaf(int32_t c) const {
        return c < 0 || (firstTri != nullptr && __float_as_int(boxes[2 * c + 1].w) > 0);
    }
    __device__ __forceinline__ int32_t leaf_code(int32_t c) const {
        if (c < 0) return pack_leaf(triPos ? triPos[~c] : ~c, 1);
        return pack_leaf(firstTri[c], __float_as_int(boxes[2 * c + 1].w));
    }
};

__global__ void __launch_bounds__(256) k_emit_nodes(int n, const int32_t* __restrict__ children,
                                                    const float4* __restrict__ boxes,
                                                    const float* __restrict__ grid, const int32_t* __restrict__ order,
                                                    LeafView lv, uint4* __restrict__ nodes) {
    const int src = blockIdx.x * blockDim.x + threadIdx.x;
    if (src >= n - 1) return;
    const int32_t cl = children[2 * src], cr = children[2 * src + 1];
    const int el = cl >= 0 ? cl : (n - 1 + ~cl), er = cr >= 0 ? cr : (n - 1 + ~cr);
    const float4 llo = boxes[2 * el], lhi = boxes[2 * el + 1];
    const float4 rlo = boxes[2 * er], rhi = boxes[2 * er + 1];
    // `order` (optional) relabels inner nodes; the root keeps index 0
    const int i = order ? order[src] : src;
    const int32_t pl = lv.is_leaf(cl) ? lv.leaf_code(cl) : (order ? order[cl] : cl);
    const int32_t pr = lv.is_leaf(cr) ? lv.leaf_code(cr) : (order ? order[cr] : cr);
    // outward rounding with a guard band (kGuardCells) against the rounding of the scaling itself and of the slab test
    auto qlo = [&](float v, int k) {
        const float c = floorf((v - grid[k]) * grid[3 + k] - kGuardCells);
        return (uint32_t)fminf(fmaxf(c, 0.0f), 65535.0f);
    };
    auto qhi = [&](float v, int k) {
        const float c = ceilf((v - grid[k]) * grid[3 + k] + kGuardCells);
        return (uint32_t)fminf(fmaxf(c, 0.0f), 65535.0f);
    };
    // one word per axis: lower plane | extent << 16 (rt_scene.cuh, slab1)
    auto pack = [&](float lo, float hi, int k) {
        const uint32_t l = qlo(lo, k), h = qhi(hi, k);
        return l | ((h - l) << 16);
    };
    uint4 a, b;
    a.x = pack(llo.x, lhi.x, 0);
    a.y = pack(llo.y, lhi.y, 1);
    a.z = pack(llo.z, lhi.z, 2);
    a.w = pack(rlo.x, rhi.x, 0);
    b.x = pack(rlo.y, rhi.y, 1);
    b.y = pack(rlo.z, rhi.z, 2);
    b.z = (uint32_t)pl;
    b.w = (uint32_t)pr;
    nodes[2 * i + 0] = a;
    nodes[2 * i + 1] = b;
}

// ---------------------------------------------------------------------------------------------
// 4-wide nodes, collapsed from the binary tree level by level: every queue entry (binary inner node, wide index)
// starts from the node's two children and opens, at most twice, the inner child with the largest surface area.
// Inner slots get a wide index and go to the next level's queue; leaf slots keep their packed leaf code; unused
// slots carry the degenerate box at the far grid corner and the leaf code of triangle 0 (no box is unhittable; a ray
// through that corner merely tests one triangle more).
// 64 bytes per node = 4 x (3 words of lo | extent << 16) + 4 children.
// Numbering depends on atomics (topology does not), which is harmless: the closest-hit rule makes the image
// independent of the hierarchy's layout.
// Counters (uint32, in the dead histogram buffer): cnt[0..2] = queue sizes, rotating (level L reads cnt[L % 3],
// appends to cnt[(L + 1) % 3] and clears cnt[(L + 2) % 3] for the level after next), cnt[3] = levels that had work.
// wide[0] = wide nodes allocated, wide[1] = worst-case number of traversal-stack entries: a visit of a node with k
// children pushes at most k - 1 of them, so the deepest stack any ray can build is the largest sum of (k - 1)
// along a root-to-leaf path; needOf[wide index] carries that sum down the levels.
__global__ void __launch_bounds__(256) k_collapse4(int n, int level, const int32_t* __restrict__ children,
                                                   const float4* __restrict__ boxes, const float* __restrict__ grid,
                                                   const int2* __restrict__ qin, int2* __restrict__ qout,
                                                   uint32_t* __restrict__ cnt, uint32_t* __restrict__ wide,
                                                   uint32_t* __restrict__ needOf, LeafView lv,
                                                   uint4* __restrict__ nodes4) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t count = cnt[level % 3];
    uint32_t* qoutCount = cnt + (level + 1) % 3;
    if (i == 0) {
        cnt[(level + 2) % 3] = 0u;
        if (count > 0u) cnt[3] = (uint32_t)level + 1u;
    }
    if (i >= count) return;
    const int2 e = qin[i];
    int32_t slot[4] = {children[2 * e.x], children[2 * e.x + 1], -1, -1};
    int cnt4 = 2;
    auto ent = [&](int32_t c) { return c >= 0 ? c : (n - 1 + ~c); };
    auto area = [&](int32_t c) {
        const float4 lo = boxes[2 * ent(c)], hi = boxes[2 * ent(c) + 1];
        const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
        return dx * dy + dy * dz + dz * dx;
    };
    for (int round = 0; round < 2; round++) {
        int best = -1;
        float bestA = -1.0f;
        for (int k = 0; k < cnt4; k++)
            if (!lv.is_leaf(slot[k])) {
                const float a = area(slot[k]);
                if (a > bestA) { bestA = a; best = k; }
            }
        if (best < 0) break;
        const int32_t open = slot[best];
        slot[best] = children[2 * open];
        slot[cnt4++] = children[2 * open + 1];
    }
    const uint32_t need = needOf[e.y] + (uint32_t)(cnt4 - 1);
    atomicMax(&wide[1], need);
    auto qlo = [&](float v, int k) {
        const float c = floorf((v - grid[k]) * grid[3 + k] - kGuardCells);
        return (uint32_t)fminf(fmaxf(c, 0.0f), 65535.0f);
    };
    auto qhi = [&](float v, int k) {
        const float c = ceilf((v - grid[k]) * grid[3 + k] + kGuardCells);
        return (uint32_t)fminf(fmaxf(c, 0.0f), 65535.0f);
    };
    uint32_t w[16];
    for (int k = 0; k < 4; k++) {
        if (k < cnt4) {
            const float4 lo = boxes[2 * ent(slot[k])], hi = boxes[2 * ent(slot[k]) + 1];
            const uint32_t lx = qlo(lo.x, 0), ly = qlo(lo.y, 1), lz = qlo(lo.z, 2);
            w[3 * k + 0] = lx | ((qhi(hi.x, 0) - lx) << 16);  // lower plane | extent << 16 (rt_scene.cuh, slab1)
            w[3 * k + 1] = ly | ((qhi(hi.y, 1) - ly) << 16);
            w[3 * k + 2] = lz | ((qhi(hi.z, 2) - lz) << 16);
            int32_t ref;
            if (!lv.is_leaf(slot[k])) {
                ref = (int32_t)atomicAdd(&wide[0], 1u);
                needOf[ref] = need;
                qout[atomicAdd(qoutCount, 1u)] = make_int2(slot[k], ref);
            } else {
                ref = lv.leaf_code(slot[k]);
            }
            w[12 + k] = (uint32_t)ref;
        } else {
            w[3 * k + 0] = w[3 * k + 1] = w[3 * k + 2] = 0x0000ffffu;  // lo = 65535, extent 0
            w[12 + k] = (uint32_t)pack_leaf(0, 1);
        }
    }
    uint4* dst = nodes4 + 4 * (size_t)e.y;
    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    dst[2] = make_uint4(w[8], w[9], w[10], w[11]);
    dst[3] = make_uint4(w[12], w[13], w[14], w[15]);
}
__global__ void k_collapse_init(int2* q, uint32_t* cnt, uint32_t* wide, uint32_t* needOf) {
    if (threadIdx.x == 0) {
        q[0] = make_int2(0, 0);  // the binary root becomes wide node 0
        cnt[0] = 1u;             // entries in the level-0 queue
        cnt[1] = 0u;
        cnt[2] = 0u;
        cnt[3] = 0u;             // levels
        wide[0] = 1u;            // wide nodes allocated
        wide[1] = 0u;            // worst-case stack entries
        needOf[0] = 0u;
    }
}
__global__ void k_set_word(uint32_t* p, uint32_t v) {
    if (threadIdx.x == 0) *p = v;
}

// Sorted triangle records.  e0, e1 and N are computed with exactly the operations of
// compute.glsl:307-309 (and -fmad=false), so precomputing them changes no bit of any hit.
__global__ void __launch_bounds__(256) k_emit_tris(const rt_triangle* __restrict__ tris,
                                                   const uint32_t* __restrict__ sortedIdx,
                                                   const int32_t* __restrict__ triPos, int n,
                                                   float4* __restrict__ geom, float4* __restrict__ shade,
                                                   int32_t* __restrict__ orig) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;  // position in Morton order
    if (m >= n) return;
    const uint32_t src = sortedIdx[m];
    const int s = triPos ? triPos[m] : m;                  // record slot: depth-first order of the leaves
    const rt_triangle& t = tris[src];
    const V3 a = v3(t.a), b = v3(t.b), c = v3(t.c);
    const V3 e0 = b - a, e1 = c - a;
    const V3 N = cross(e0, e1);
    geom[4 * s + 0] = make_float4(a.x, a.y, a.z, e0.x);
    geom[4 * s + 1] = make_float4(e0.y, e0.z, e1.x, e1.y);
    geom[4 * s + 2] = make_float4(e1.z, N.x, N.y, N.z);
    const V3 nrm = normalize(N);  // compute.glsl:331, the very expression k_shade used to evaluate per hit
    geom[4 * s + 3] = make_float4(nrm.x, nrm.y, nrm.z, __int_as_float(t.materialIndex));
    shade[2 * s + 0] = make_float4(t.aTex[0], t.aTex[1], t.bTex[0], t.bTex[1]);
    shade[2 * s + 1] = make_float4(t.cTex[0], t.cTex[1], __int_as_float(t.materialIndex), __int_as_float((int32_t)src));
    orig[s] = (int32_t)src;
}

__global__ void k_iota(uint32_t* v, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

// ---------------------------------------------------------------------------------------------
// Host driver.  Depth, error flags and the wide-tree counters stay on the device for rt_scene_build to read.
cudaError_t build_lbvh(const BuildArgs& a, cudaStream_t st, uint64_t* launches) {
    const int n = a.n;
    auto nb = [](long long count, int per) { return (int)((count + per - 1) / per); };
    uint64_t L = 0;
    // RT_BUILD_DEBUG=1: synchronise after every launch and name the first kernel that fails
    static const bool debug = getenv("RT_BUILD_DEBUG") != nullptr;
#define RT_DBG()                                                                                            \
    do {                                                                                                    \
        if (debug) {                                                                                        \
            cudaError_t de = cudaStreamSynchronize(st);                                                     \
            if (de != cudaSuccess) {                                                                        \
                fprintf(stderr, "build_lbvh: launch before line %d failed: %s\n", __LINE__, cudaGetErrorString(de)); \
                return de;                                                                                  \
            }                                                                                               \
        }                                                                                                   \
    } while (0)
    uint32_t* maxDepth = a.status + kBuildDepth;
    cudaMemsetAsync(a.status, 0, kBuildStatusWords * sizeof(uint32_t), st);
    k_init_bounds<<<1, 32, 0, st>>>(a.bounds); L++; RT_DBG();
    k_tri_bounds<<<min(nb(n, 256), a.sm_count * 8), 256, 0, st>>>(a.tris, n, a.centroid, a.bounds, a.status); L++; RT_DBG();
    if (n >= 2) {
        k_morton<<<nb(n, 256), 256, 0, st>>>(a.centroid, n, a.bounds, a.keys[0], a.vals[0]); L++; RT_DBG();
        const int nblocks = nb(n, kSortTile);
        int cur = 0;
        for (int pass = 0; pass < 8; pass++) {
            const int shift = pass * 8;
            k_hist<<<nblocks, kSortThreads, 0, st>>>(a.keys[cur], n, shift, a.hist, nblocks); L++; RT_DBG();
            k_scan<<<1, 1024, 0, st>>>(a.hist, 256 * nblocks); L++; RT_DBG();
            k_scatter<<<nblocks, kSortThreads, 0, st>>>(a.keys[cur], a.vals[cur], a.keys[cur ^ 1],
                                                        a.vals[cur ^ 1], n, shift, a.hist, nblocks); L++; RT_DBG();
            cur ^= 1;
        }
        // 8 passes: the result is back in buffer 0
    } else {
        k_iota<<<1, 32, 0, st>>>(a.vals[0], n); L++; RT_DBG();
    }
    int32_t* order = nullptr;
    int32_t *firstTri = nullptr, *triPos = nullptr;
    if (n >= 2 && a.use_ploc) {
        // scratch: the sort's second key/value buffers are free now
        int32_t* cluster[2] = {reinterpret_cast<int32_t*>(a.vals[1]), a.parent};
        int32_t* nn = a.parent + n;                      // parent has 2n entries
        uint32_t* height = a.nodeDepth;                   // 2n - 1 entries
        int32_t* parentOf = reinterpret_cast<int32_t*>(a.centroid);     // centroids are dead after k_morton: 16n bytes
        uint32_t* innerCount = reinterpret_cast<uint32_t*>(a.centroid) + n;
        int32_t* leafParent = reinterpret_cast<int32_t*>(a.flags);      // n + 1 words, free since the scan moved into the merge kernel
        const LeafPolicy pol{0.35f, 4};
        const int radius = kPlocRadiusDefault;
        uint32_t* ctl = a.hist;                           // the histograms are dead after the sort
        unsigned long long* tileState = reinterpret_cast<unsigned long long*>(a.hist + kCtlWords);
        k_ploc_init<<<nb(n, 256), 256, 0, st>>>(a.tris, a.vals[0], n, a.bounds, a.boxes, cluster[0], height); L++; RT_DBG();
        k_ploc_ctl_init<<<1, 32, 0, st>>>(ctl, n); L++; RT_DBG();
        // Rounds are enqueued in chunks without the host knowing the cluster count (kernels read it from `ctl`;
        // grids are sized for the count at the start of the chunk, surplus blocks exit at once); after each chunk
        // the single-block tail gets a chance and the host reads back two words.
        int round = 0, chunk = 4;
        uint32_t m = (uint32_t)n;
        const int kMaxGlobalRounds = 1024;
        while (m > 1u) {
            if (m > (uint32_t)kPlocTailMax) {
                for (int k = 0; k < chunk; k++, round++) {
                    k_ploc_nn<<<nb(m, 256), 256, 0, st>>>(n, round, ctl, tileState, cluster[0], cluster[1], a.boxes, nn, radius); L++; RT_DBG();
                    k_ploc_merge_scan<<<nb(m, kPlocTile), 256, 0, st>>>(n, round, ctl, tileState, cluster[0],
                                                                         cluster[1], nn, a.boxes, a.children,
                                                                         height, parentOf, innerCount, leafParent, pol, a.status); L++; RT_DBG();
                }
                chunk = min(chunk * 2, 64);
            }
            k_ploc_tail<<<1, 1024, 0, st>>>(n, round, ctl, cluster[0], cluster[1], a.boxes, a.children, height, parentOf,
                                            innerCount, leafParent, pol, a.status, radius); L++; RT_DBG();
            uint32_t state[2];
            cudaMemcpyAsync(state, ctl + 4 * (round & 1), sizeof state, cudaMemcpyDeviceToHost, st);
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return e;
            m = state[0];
            if (m > 1u && round >= kMaxGlobalRounds) {  // runs of identical boxes merge one pair per round: not worth waiting for
                k_set_word<<<1, 32, 0, st>>>(a.status + kBuildPlocStuck, 1u); L++; RT_DBG();
                m = 0u;
            }
        }
        k_ploc_depth<<<1, 32, 0, st>>>(height, maxDepth); L++; RT_DBG();
        // depth-first positions: of the inner nodes (their index in memory), of the triangles in
        // front of every subtree, and of every triangle (the order of the triangle records: leaves are contiguous runs)
        order = reinterpret_cast<int32_t*>(a.centroid) + 2 * (size_t)n;
        firstTri = reinterpret_cast<int32_t*>(a.centroid) + 3 * (size_t)n;
        triPos = reinterpret_cast<int32_t*>(a.vals[1]);  // the cluster list that lived here is dead
        k_dfs_order<<<nb(n - 1, 256), 256, 0, st>>>(n, a.children, parentOf, innerCount, order, firstTri); L++; RT_DBG();
        k_tri_order<<<nb(n, 256), 256, 0, st>>>(n, a.children, parentOf, leafParent, innerCount, triPos); L++; RT_DBG();
    } else {
        if (n >= 2) {
            k_hierarchy<<<nb(n - 1, 256), 256, 0, st>>>(a.keys[0], n, a.children, a.parent); L++; RT_DBG();
            cudaMemsetAsync(a.flags, 0, sizeof(uint32_t) * (size_t)(n - 1), st);
            cudaMemsetAsync(a.nodeDepth, 0, sizeof(uint32_t) * (size_t)(n - 1), st);
        }
        k_refit<<<nb(n, 256), 256, 0, st>>>(a.tris, a.vals[0], n, a.bounds, a.children, a.parent, a.boxes, a.flags,
                                            a.nodeDepth, maxDepth); L++; RT_DBG();
    }
    k_grid<<<1, 32, 0, st>>>(a.bounds, a.grid); L++; RT_DBG();
    const LeafView lv{a.boxes, triPos, firstTri, n};
    if (n >= 2) { k_emit_nodes<<<nb(n - 1, 256), 256, 0, st>>>(n, a.children, a.boxes, a.grid, order, lv, a.nodes); L++; RT_DBG(); }
    if (n >= 2 && a.nodes4) {
        // queues in the two key buffers of the sort (n int2 each, dead by now); counters behind the PLOC control
        // block; per-node stack need in the height array (dead after k_ploc_depth / k_refit)
        int2* q[2] = {reinterpret_cast<int2*>(a.keys[0]), reinterpret_cast<int2*>(a.keys[1])};
        uint32_t* cnt = a.hist + 32;
        uint32_t* needOf = a.nodeDepth;
        k_collapse_init<<<1, 32, 0, st>>>(q[0], cnt, a.wide_count, needOf); L++; RT_DBG();
        // levels are enqueued 16 at a time with grids sized by the bound min(4^level, n - 1) on the queue length;
        // an empty level is a no-op, and after each group the host reads one word to see whether work remains
        int level = 0;
        uint32_t pending = 1u;
        while (pending > 0u) {
            for (int k = 0; k < 16; k++, level++) {
                const long long bound = level < 13 ? (1ll << (2 * level)) : (long long)n;
                const long long cap = bound < (long long)(n - 1) ? bound : (long long)(n - 1);
                k_collapse4<<<nb(cap, 256), 256, 0, st>>>(n, level, a.children, a.boxes, a.grid, q[level & 1],
                                                          q[(level + 1) & 1], cnt, a.wide_count, needOf, lv, a.nodes4); L++; RT_DBG();
            }
            cudaMemcpyAsync(&pending, cnt + level % 3, sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return e;
        }
        uint32_t levels = 0;
        cudaMemcpyAsync(&levels, cnt + 3, sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        if (a.wide_levels) *a.wide_levels = (int)levels;
    }
    k_emit_tris<<<nb(n, 256), 256, 0, st>>>(a.tris, a.vals[0], triPos, n, a.geom, a.shade, a.orig); L++; RT_DBG();
    if (launches) *launches += L;
#undef RT_DBG
    return cudaGetLastError();
}

// sort histograms (+1: k_scan stores the total); the same words later hold the PLOC control block, the tile
// states of its scan (one uint64 per kPlocTile clusters) and the collapse counters
size_t build_scratch_words(int n) {
    const size_t sortWords = (size_t)256 * ((n + kSortTile - 1) / kSortTile) + 1;
    const size_t plocWords = (size_t)kCtlWords + 2 * ((size_t)(n + kPlocTile - 1) / kPlocTile + 1) + 64;
    return sortWords > plocWords ? sortWords : plocWords;
}

}  // namespace rt
