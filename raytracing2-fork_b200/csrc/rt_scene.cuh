// rt_scene.cuh — device-side scene layout and the closest-hit traversal shared by every kernel.
//
// HBM layout (DESIGN.md §3).  ncu showed the traversal kernel bound by the L1TEX data pipe
// (l1tex__data_pipe_lsu_wavefronts 89-95 % of peak): a gather where every lane reads its own node is
// served at ~16 bytes per lane per wavefront, so the only lever is BYTES PER VISIT.
//   nodes    : 32 B per inner node = ONE 256-bit load (LDG.E.256 on sm_100a).  Both child boxes
//              live in the parent, quantised to 16 bits per plane on a global grid over the padded
//              scene box and rounded OUTWARD (the boxes only prune, so a larger box is always
//              safe; triangle tests stay exact binary32).  Per axis one word = lower plane | EXTENT << 16
//              (extent = upper - lower plane, in cells): the slab test then needs no min / max to order the
//              two planes of an axis (slab1 below):
//                w0..w2 = left  child (lo.x | ext.x << 16, lo.y | ext.y << 16, lo.z | ext.z << 16)
//                w3..w5 = right child, w6 = left, w7 = right
//              child >= 0: inner node index; child < 0: leaf, ~child = first | (count-1) << 27.
//              (The reference re-reads the 48-byte parent and then two 48-byte children per visit:
//              144 B, compute.glsl:425,443-444.)
//   nodes4   : 64 B per 4-wide node (two 256-bit loads), collapsed from the binary tree by k_collapse4: four child
//              boxes w0..w11 (three words each, same quantisation), four children w12..w15.  k_extend walks these by
//              default; the binary nodes serve the preview kernel, RT_BVH_WIDTH=2 and the deep-tree fallback.
//   tri_geom : 64 B stride per sorted triangle; traversal reads the first 48 B = a, e0 = b-a,
//              e1 = c-a, N = cross(e0,e1), precomputed with the very operations
//              compute.glsl:307-309 performs per test, so every bit of dst,u,v is unchanged
//   tri_shade: 32 B per sorted triangle = aTex,bTex,cTex, materialIndex, original index
//   tri_orig : 4 B per sorted triangle, the index in the caller's array (tie-break + reported id)
#pragma once
#include "rt_math.cuh"

namespace rt {

struct SceneView {
    const uint4* __restrict__ nodes;       // 2 per inner node (32 B, 32-byte aligned)
    const uint4* __restrict__ nodes4;      // 4 per 4-wide node (64 B), or NULL (RT_BVH_WIDTH=4 builds them for k_extend)
    const float4* __restrict__ tri_geom;   // 4 per sorted triangle (64 B, 32-byte aligned)
    const float4* __restrict__ tri_shade;  // 2 per sorted triangle
    const int32_t* __restrict__ tri_orig;
    const float4* __restrict__ materials;  // 6 float4 per material (the 96-byte reference struct)
    const uint8_t* tex_px[5];
    int32_t tex_w[5], tex_h[5], tex_ch[5];
    int32_t num_tris;
    int32_t num_nodes4;    // 4-wide nodes behind `nodes4`
    int32_t num_materials;
    int32_t root_is_leaf;  // scenes with a single triangle have no inner node
    float grid_lo[3];      // world position of quantised coordinate 0
    float grid_inv[3];     // cells per world unit (65535 cells span the padded scene box)
};

struct HitRec {
    float t;       // 1e38f = miss
    float u, v;
    int32_t slot;  // sorted slot, -1 = miss
};

// traversal stack entries per ray: 16 in shared memory (k_extend), the rest in local memory.  rt_scene_build checks the
// exact worst case of the tree it built against this (binary: depth; 4-wide: sum of children-1 along the deepest path).
constexpr int kStackSize = 256;
// outward rounding margin of the quantised planes, in grid cells (bvh_build.cu k_emit_nodes; bound in slab1 below)
constexpr float kGuardCells = 0.125f;

// 256-bit read-only global load (sm_100a: LDG.E.ENL2.256.CONSTANT): one instruction, one L1TEX
// wavefront per lane for 32 bytes, where four 128-bit loads of a 64-byte record would cost four.
// (L1 eviction-priority hints on this load and on load_tri's measured neutral or slower: profiles/r2_final_ab.txt.)
__device__ __forceinline__ void ldg256u(const void* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p));
}
// exact uint16 -> float with I2F.U16: one instruction that reads the half register directly, but on the XU pipe,
// 16 lanes / clk / SM (tools/microbench.cu: 4.5 T/s against 17.8 T/s FFMA instructions).  A 4-wide visit converts 24
// planes; ncu round 2 had XU 54 % busy, the busiest pipe relative to its rate.  Splicing the 16 bits into the mantissa
// of 2^23 and subtracting 2^23 moves the work to the ALU and FMA pipes, but costs a second instruction per plane, and
// the kernel is bound by issue slots: that byte-permute variant measured slower for either half and for both
// (config 2, 5580-5787 vs 5880 Mrays/s, profiles/r2_deq_ab.txt).
__device__ __forceinline__ float q_lo(uint32_t w) { return (float)(uint16_t)(w & 0xffffu); }
__device__ __forceinline__ float q_hi(uint32_t w) { return (float)(uint16_t)(w >> 16); }

// The ray in grid coordinates: per-axis scaling of origin and direction leaves t unchanged.
struct GridRay {
    float ox, oy, oz;     // -(o - grid_lo) * grid_inv * i: the constant term of t = q * i + c
    float ix, iy, iz;     // 1 / (d * grid_inv), clamped to +-1e28
    float nx, ny, nz;     // min(i, 0): the slope that takes the lower plane's t to the NEAR plane's
};
__device__ __forceinline__ GridRay make_grid_ray(const SceneView& sc, V3 o, V3 d) {
    GridRay g;
    g.ox = (o.x - sc.grid_lo[0]) * sc.grid_inv[0];
    g.oy = (o.y - sc.grid_lo[1]) * sc.grid_inv[1];
    g.oz = (o.z - sc.grid_lo[2]) * sc.grid_inv[2];
    g.ix = 1.0f / (d.x * sc.grid_inv[0]);
    g.iy = 1.0f / (d.y * sc.grid_inv[1]);
    g.iz = 1.0f / (d.z * sc.grid_inv[2]);
    // finite slopes keep q*i + c free of inf - inf; a ray parallel to a slab then decides by the sign of
    // (q - o) * 1e28, which the builder's guard band keeps right (kGuardCells)
    g.ix = fminf(fmaxf(g.ix, -1e28f), 1e28f);
    g.iy = fminf(fmaxf(g.iy, -1e28f), 1e28f);
    g.iz = fminf(fmaxf(g.iz, -1e28f), 1e28f);
    g.ox = -g.ox * g.ix;
    g.oy = -g.oy * g.iy;
    g.oz = -g.oz * g.iz;
    g.nx = fminf(g.ix, 0.0f);
    g.ny = fminf(g.iy, 0.0f);
    g.nz = fminf(g.iz, 0.0f);
    return g;
}
// Slab test against a quantised box, three FFMAs per axis and NO per-axis min / max (ncu, round 2: the ALU pipe, which
// executes FMNMX / SEL / ISETP at half the rate of the FMA pipe, was the busiest pipe of k_extend at 62 %, the FMA pipe
// idled at 20 %).  With lo the lower plane and ext >= 0 the extent of the box along the axis, both in cells:
//     t_lo   = fma(lo, i, c)            the ray parameter at the lower plane
//     t_near = fma(ext, min(i, 0), t_lo)   = t_lo for i >= 0, the upper plane's parameter for i < 0
//     t_far  = fma(ext, |i|, t_near)       (|.| is a free operand modifier)
// Conservativeness.  u = 2^-24, Q = 65535 cells, O = |origin| in cells.  The grid transform of the origin costs 2u O,
// the slope 2u relative, the constant term c = -o i therefore 5u O |i|; t_lo then carries |i| u (3 lo + 6 O), t_near
// |i| u (6 Q + 7 O) and t_far |i| u (9 Q + 8 O): a plane is displaced by at most u (9 Q + 8 O) cells — 0.066 cell for
// an origin inside the grid, 0.10 cell at O = 140 000.  The builder rounds every plane outward by kGuardCells = 1/8
// cell (its own scaling costs another 2u Q = 0.008 cell), so for origins within ~2.1 grid extents rounding can never
// cull a true hit.  For origins farther out (WIDEN) the far side is widened by 2e-6 relative = 33u |t_far|, which
// exceeds the sum of both sides' errors, u (15 Q + 15 O), once O > Q.  Slopes are clamped to +-1e28: no inf - inf
// for rays parallel to a slab.
// WIDEN = false drops that widening: every bounce ray starts on a surface of the scene, i.e. inside the grid, and so
// does a camera that stands inside or near the scene box — k_extend is instantiated both ways and the host picks per
// launch (rt_api.cu: widen_needed).
constexpr float kWidenFar = 1.000002f;
constexpr float kSlabMiss = 3.0e38f;
__device__ __forceinline__ void slab_axis(uint32_t w, float c, float i, float n, float& tNear, float& tFar) {
    const float tLo = __fmaf_rn(q_lo(w), i, c);
    const float ext = q_hi(w);
    tNear = __fmaf_rn(ext, n, tLo);
    tFar = __fmaf_rn(ext, fabsf(i), tNear);
}
// One slab test: entry distance, or kSlabMiss.
template <bool WIDEN = true>
__device__ __forceinline__ float slab1(uint32_t wx, uint32_t wy, uint32_t wz, const GridRay& g, float bestT) {
    float nx, fx, ny, fy, nz, fz;
    slab_axis(wx, g.ox, g.ix, g.nx, nx, fx);
    slab_axis(wy, g.oy, g.iy, g.ny, ny, fy);
    slab_axis(wz, g.oz, g.iz, g.nz, nz, fz);
    const float tn = fmaxf(fmaxf(nx, ny), fmaxf(nz, 0.0f));
    float tf = fminf(fminf(fx, fy), fminf(fz, bestT));
    if (WIDEN) tf *= kWidenFar;
    return tn <= tf ? tn : kSlabMiss;
}
// Two slab tests against the child boxes of a binary node.
template <bool WIDEN = true>
__device__ __forceinline__ void slab2(const uint32_t (&w)[8], const GridRay& g, float bestT, float& lNear,
                                      float& rNear, bool& hitL, bool& hitR) {
    const float l = slab1<WIDEN>(w[0], w[1], w[2], g, bestT);
    const float r = slab1<WIDEN>(w[3], w[4], w[5], g, bestT);
    hitL = l < kSlabMiss;
    hitR = r < kSlabMiss;
    lNear = l;
    rNear = r;
}
// first 48 bytes of a triangle record: a, e0, e1, N
struct TriGeom {
    V3 a, e0, e1, N;
};
__device__ __forceinline__ TriGeom load_tri(const SceneView& sc, int32_t s) {
    float g[8];
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(g[0]), "=f"(g[1]), "=f"(g[2]), "=f"(g[3]), "=f"(g[4]), "=f"(g[5]), "=f"(g[6]), "=f"(g[7])
                 : "l"(sc.tri_geom + 4 * s));
    float4 h;
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(h.x), "=f"(h.y), "=f"(h.z), "=f"(h.w)
                 : "l"(sc.tri_geom + 4 * s + 2));
    TriGeom t;
    t.a = v3(g[0], g[1], g[2]);
    t.e0 = v3(g[3], g[4], g[5]);
    t.e1 = v3(g[6], g[7], h.x);
    t.N = v3(h.y, h.z, h.w);
    return t;
}
__device__ __forceinline__ void ldg256(const void* p, float (&v)[8]) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}
constexpr float kMissT = 1e38f;

// compute.glsl:302-340 on the precomputed (a, e0, e1, N).  Returns true on a hit and the same
// dst/u/v bits the reference expression order produces.
// tMax: a candidate farther than the best hit so far cannot win; leaving before the barycentrics changes no result.
__device__ __forceinline__ bool ray_triangle(V3 o, V3 d, V3 a, V3 e0, V3 e1, V3 N, float& dst,
                                             float& u, float& v, float tMax = 3.4e38f) {
    const float det = -dot(d, N);
    if ((det < 1e-10f && det > -1e-10f) || det < 0.0f) return false;
    const float invDet = 1.0f / det;
    const V3 ao = o - a;
    dst = dot(ao, N) * invDet;
    if (dst <= 1e-6f || dst > tMax) return false;
    const V3 dao = cross(d, ao);
    u = -dot(e1, dao) * invDet;
    v = dot(e0, dao) * invDet;
    if (u < 0.0f || v < 0.0f || 1.0f - u - v < 0.0f) return false;
    return true;
}

// Leaf children are packed into one negative int: child = ~(first | (count-1) << 27).
constexpr int kLeafCountShift = 27;
constexpr int32_t kLeafFirstMask = (1 << kLeafCountShift) - 1;
__host__ __device__ __forceinline__ int32_t pack_leaf(int32_t first, int32_t count) {
    return ~(first | ((count - 1) << kLeafCountShift));
}

// Closest hit = min dst, ties → lowest ORIGINAL triangle index (SURVEY A.6).  The BVH only prunes:
// a subtree is skipped when its (conservatively widened) slab interval cannot contain a hit with
// t <= best, so the result equals the exhaustive minimum over all triangles regardless of the
// hierarchy or the visiting order.
__device__ __forceinline__ HitRec closest_hit(const SceneView& sc, V3 o, V3 d) {
    HitRec best;
    best.t = kMissT;
    best.u = 0.0f;
    best.v = 0.0f;
    best.slot = -1;
    int32_t bestOrig = 0x7fffffff;
    if (sc.num_tris <= 0) return best;

    const GridRay g = make_grid_ray(sc, o, d);
    const float kWiden = kWidenFar;

    int32_t stack[kStackSize];
    float tstack[kStackSize];
    int sp = 0;
    int32_t cur = sc.root_is_leaf ? pack_leaf(0, sc.num_tris) : 0;

    for (;;) {
        if (cur >= 0) {
            uint32_t w[8];
            ldg256u(sc.nodes + 2 * cur, w);
            float lNear, rNear;
            bool hitL, hitR;
            slab2(w, g, best.t, lNear, rNear, hitL, hitR);
            const int32_t cl = (int32_t)w[6], cr = (int32_t)w[7];
            if (hitL && hitR) {
                const bool leftFirst = lNear <= rNear;
                stack[sp] = leftFirst ? cr : cl;
                tstack[sp] = leftFirst ? rNear : lNear;
                sp++;
                cur = leftFirst ? cl : cr;
                continue;
            } else if (hitL) {
                cur = cl;
                continue;
            } else if (hitR) {
                cur = cr;
                continue;
            }
        } else {
            const int32_t packed = ~cur;
            const int32_t first = packed & kLeafFirstMask;
            const int32_t count = (packed >> kLeafCountShift) + 1;
            for (int32_t s = first; s < first + count; s++) {
                const TriGeom tg = load_tri(sc, s);
                float dst, u, v;
                if (ray_triangle(o, d, tg.a, tg.e0, tg.e1, tg.N, dst, u, v)) {
                    if (dst <= best.t && dst < kMissT) {
                        const int32_t orig = __ldg(&sc.tri_orig[s]);
                        if (dst < best.t || orig < bestOrig) {
                            best.t = dst;
                            best.u = u;
                            best.v = v;
                            best.slot = s;
                            bestOrig = orig;
                        }
                    }
                }
            }
        }
        // pop the next subtree that can still hold a hit with t <= best
        bool got = false;
        while (sp > 0) {
            --sp;
            if (tstack[sp] <= best.t * kWiden) {
                cur = stack[sp];
                got = true;
                break;
            }
        }
        if (!got) break;
    }
    return best;
}

}  // namespace rt
