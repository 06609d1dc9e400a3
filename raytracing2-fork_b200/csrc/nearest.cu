// nearest.cu — nearest-triangle (closest-point) queries on device memory: k_nearest<COUNT, WIDE>.
//
// For every query point p and optional radius r: among the triangles with dist(p, T) < min(r, 1e38), the one with
// the smallest distance, exact ties to the lowest original id; its distance, barycentrics (u, v) of the closest
// point a + e0 u + e1 v and that point.  A miss writes -1 / 1e38 / 0 / 0 and (0, 0, 0).  A NaN, zero or negative
// radius and a point with a non-finite coordinate never hit and are not traversed.  DESIGN.md §5, "Nearest-triangle
// queries".
#include "rt_internal.h"

namespace rt {

namespace {

constexpr int kNearBlock = 128;

__device__ __forceinline__ float clamp01(float x) {
    x = x > 0.0f ? x : 0.0f;  // NaN -> 0
    return x < 1.0f ? x : 1.0f;
}

// Distance from the point to the closed triangle (a, e0 = b - a, e1 = c - a), the exact binary32 twin of the CPU
// reference's pointTriangle (tests/native/nearest_oracle.cpp; -fmad=false here, -ffp-contract=off there; keep the two
// in step).
// Ericson, Real-Time Collision Detection §5.1.5, restated on the stored (a, e0, e1):
//   ap = p - a, bp = ap - e0, cp = ap - e1
//   d1 = dot(e0, ap), d2 = dot(e1, ap), d3 = dot(e0, bp), d4 = dot(e1, bp), d5 = dot(e0, cp), d6 = dot(e1, cp)
//   A: d1 <= 0 && d2 <= 0                                   -> (u, v) = (0, 0)
//   B: d3 >= 0 && d4 <= d3                                  -> (1, 0)
//   vc = d1 * d4 - d3 * d2
//   AB: vc <= 0 && d1 >= 0 && d3 <= 0, t = d1 / (d1 - d3)   -> (t, 0)
//   C: d6 >= 0 && d5 <= d6                                  -> (0, 1)
//   vb = d5 * d2 - d1 * d6
//   AC: vb <= 0 && d2 >= 0 && d6 <= 0, t = d2 / (d2 - d6)   -> (0, t)
//   va = d3 * d6 - d5 * d4
//   BC: va <= 0 && d4 - d3 >= 0 && d5 - d6 >= 0, t = (d4 - d3) / ((d4 - d3) + (d5 - d6))   -> (1 - t, t)
//   face: va > 0 && vb > 0 && vc > 0, s = (va + vb) + vc finite, k = 1 / s   -> (vb * k, vc * k),
//         final if s >= (dot(e0, e0) * dot(e1, e1)) / 64
//   otherwise: the nearest of the face point (if any) and the segment points AB, AC, BC, in that order, the first
//              winning an exact tie of dot(ap - q, ap - q); each segment t = clamp01(dot(x, e) / dot(e, e)) with
//              (x, e) = (ap, e0), (ap, e1), (bp, e1 - e0), or t = 0 when dot(e, e) is not > 0
//   q = e0 * u + e1 * v, dist = sqrt(dot(ap - q, ap - q)), point = a + q
// An edge case is taken only when its quotient is defined (denominator > 0 and the quotient <= 1, which also rejects
// the NaN of inf / inf); otherwise the tests go on.  Zero-length edges, collinear and coincident vertices then reach
// the segment fallback, which never divides by zero, so the result is never NaN and is the distance to a point of
// the closed triangle, the nearest one up to rounding.
__device__ __forceinline__ void nearest_uv(V3 ap, V3 e0, V3 e1, float& u, float& v) {
    const float d1 = dot(e0, ap), d2 = dot(e1, ap);
    u = 0.0f;
    v = 0.0f;
    if (d1 <= 0.0f && d2 <= 0.0f) return;
    const V3 bp = ap - e0;
    const float d3 = dot(e0, bp), d4 = dot(e1, bp);
    if (d3 >= 0.0f && d4 <= d3) { u = 1.0f; return; }
    const float vc = d1 * d4 - d3 * d2;
    if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f) {
        const float den = d1 - d3;
        if (den > 0.0f) {
            const float t = d1 / den;
            if (t <= 1.0f) { u = t; return; }
        }
    }
    const V3 cp = ap - e1;
    const float d5 = dot(e0, cp), d6 = dot(e1, cp);
    if (d6 >= 0.0f && d5 <= d6) { v = 1.0f; return; }
    const float vb = d5 * d2 - d1 * d6;
    if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f) {
        const float den = d2 - d6;
        if (den > 0.0f) {
            const float t = d2 / den;
            if (t <= 1.0f) { v = t; return; }
        }
    }
    const float va = d3 * d6 - d5 * d4;
    const float g43 = d4 - d3, g56 = d5 - d6;
    if (va <= 0.0f && g43 >= 0.0f && g56 >= 0.0f) {
        const float den = g43 + g56;
        if (den > 0.0f) {
            const float t = g43 / den;
            if (t <= 1.0f) { u = 1.0f - t; v = t; return; }
        }
    }
    const float s = (va + vb) + vc;
    const bool face = va > 0.0f && vb > 0.0f && vc > 0.0f && s < 3.0e38f;
    if (face) {
        const float k = 1.0f / s;
        u = vb * k;
        v = vc * k;
        // s = |e0 x e1|^2 up to rounding; unless the angle at a has sin^2 >= 1/64 the weights may be rounding noise
        // (collinear vertices), and the nearest edge point competes with the face point
        if (s >= (dot(e0, e0) * dot(e1, e1)) * 0.015625f) return;
    }
    auto seg = [](V3 x, V3 e) {
        const float ee = dot(e, e);
        return ee > 0.0f ? clamp01(dot(x, e) / ee) : 0.0f;
    };
    auto dist2 = [&](float uu, float vv) {
        const V3 q = e0 * uu + e1 * vv;
        const V3 d = ap - q;
        return dot(d, d);
    };
    const float tab = seg(ap, e0), tac = seg(ap, e1), tbc = seg(bp, e1 - e0);
    float best = face ? dist2(u, v) : 3.4028235e38f;
    const float dab = dist2(tab, 0.0f);
    if (dab < best) { best = dab; u = tab; v = 0.0f; }
    const float dac = dist2(0.0f, tac);
    if (dac < best) { best = dac; u = 0.0f; v = tac; }
    const float dbc = dist2(1.0f - tbc, tbc);
    if (dbc < best) { u = 1.0f - tbc; v = tbc; }
}
__device__ __forceinline__ float point_triangle(V3 p, V3 a, V3 e0, V3 e1, float& u, float& v) {
    const V3 ap = p - a;
    nearest_uv(ap, e0, e1, u, v);
    const V3 q = e0 * u + e1 * v;
    const V3 d = ap - q;
    return sqrtf(dot(d, d));
}

// a, e0, e1: the first 36 bytes of a triangle record (one 256-bit load and one 32-bit load)
__device__ __forceinline__ void load_tri36(const SceneView& sc, int32_t s, V3& a, V3& e0, V3& e1) {
    float g[8];
    ldg256(sc.tri_geom + 4 * s, g);
    const float e1z = __ldg(reinterpret_cast<const float*>(sc.tri_geom + 4 * s + 2));
    a = v3(g[0], g[1], g[2]);
    e0 = v3(g[3], g[4], g[5]);
    e1 = v3(g[6], g[7], e1z);
}

// Lower bound on the distance from the point to anything inside one quantised child box, as a squared distance.
// pc = (p - grid_lo) * grid_inv is the point in cells, cell = 1 / grid_inv; per axis the gap to the planes [lo, lo +
// ext] in cells, times the cell size, squared and summed, then shrunk by kNearShrink2.
//
// Why the bound never exceeds the computed distance of a triangle inside the box.  u = 2^-24, Q = 65535 cells,
// ext = the largest extent of the scene box, L <= sqrt(3) ext any triangle's diameter.  Every quantised box holds the
// leaf boxes below it, each the triangle's box padded by pad >= 2e-6 ext (bvh_build.cu k_refit), and is rounded
// outward by kGuardCells = 1/8 cell, of which the builder's own scaling uses 2u Q = 0.008.  So per axis the gap from p
// to the triangle's box is at least max(0, gq + 0.117 cell + pad), gq the exact signed gap to the quantised planes.
//  - Rounding of pc: 2u |pc| cells.  For |pc| <= 2 Q (points inside or within a grid extent of the grid) that is at
//    most 0.016 cell, covered by the guard band: the computed gap is <= h = max(0, gq + 0.117 cell).  Farther out the
//    box is at least |pc| / 2 away on that axis, so the error is relative, <= 4u of the gap.
//  - The triangle side: the computed distance uses ap = p - a, q = e0 u + e1 v with (u, v) in the closed unit triangle
//    up to 2u, dot and sqrt; it is >= D (1 - 4u) - 8u L for the true distance D >= |h| + pad.  8u L <= 14u ext is
//    less than pad = 34u ext, so the computed distance is >= |h| (1 - 4u).
//  - The bound side: gap, cell size, products, squares and sums add at most 18u relative to |h|^2, and the best
//    squared distance it is compared with is rounded up (__fmul_ru).
// Together the bound squared is <= the computed squared distance times (1 + 27u) before the shrink; kNearShrink2 =
// 1 - 2^-16 (256u) covers that ten times over, and costs a relative 2^-17 of pruning distance.  The compare is
// `bound <= best`, never `<`: a box at exactly the best distance can hold a lower-id tie.  A bound or best that
// overflows to +inf compares <= +inf, so such boxes are visited (a distance whose square overflows is +inf and
// never hits).
constexpr float kNearShrink2 = 1.0f - 1.0f / 65536.0f;
struct GridPoint {
    float px, py, pz;  // the point in cells
    float cx, cy, cz;  // world units per cell
};
__device__ __forceinline__ float gap_axis(uint32_t w, float pc) {
    const float lo = q_lo(w);
    const float hi = lo + q_hi(w);  // exact: integers below 2^17
    return fmaxf(fmaxf(lo - pc, pc - hi), 0.0f);
}
__device__ __forceinline__ float box_bound2(uint32_t wx, uint32_t wy, uint32_t wz, const GridPoint& g) {
    const float gx = gap_axis(wx, g.px) * g.cx;
    const float gy = gap_axis(wy, g.py) * g.cy;
    const float gz = gap_axis(wz, g.pz) * g.cz;
    return ((gx * gx + gy * gy) + gz * gz) * kNearShrink2;
}

}  // namespace

// One thread per point, nearest child first, the stack in local memory (DESIGN.md §5 for the layout measurements).
// Stack bound: a 4-wide visit pushes at most 3 children and a binary visit 1, so the deepest stack is the
// wide_stack_need / binary depth bound that rt_scene_build checks against kStackSize before it marks a scene built.
template <bool COUNT, bool WIDE>
__global__ void __launch_bounds__(kNearBlock) k_nearest(const __grid_constant__ SceneView sc,
                                                        const __grid_constant__ NearestArgs qa, long long n,
                                                        unsigned long long* __restrict__ stats) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t visits = 0, tests = 0;
    if (i < n) {
        const V3 p = v3(qa.points[3 * i], qa.points[3 * i + 1], qa.points[3 * i + 2]);
        const float r = qa.max_dist ? qa.max_dist[i] : kMissT;
        const float limit = fminf(r, kMissT);
        // a hit needs dist < limit: start at the largest float below it and accept dist <= best (ties by id)
        float best = __int_as_float(__float_as_int(limit) - 1);
        float bu = 0.0f, bv = 0.0f;
        int32_t bestSlot = -1, bestOrig = -1;  // bestOrig: -1 = not read yet
        const bool live = sc.num_tris > 0 && r > 0.0f && isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
        if (live) {
            GridPoint g;
            g.px = (p.x - sc.grid_lo[0]) * sc.grid_inv[0];
            g.py = (p.y - sc.grid_lo[1]) * sc.grid_inv[1];
            g.pz = (p.z - sc.grid_lo[2]) * sc.grid_inv[2];
            g.cx = 1.0f / sc.grid_inv[0];
            g.cy = 1.0f / sc.grid_inv[1];
            g.cz = 1.0f / sc.grid_inv[2];
            float bestSq = __fmul_ru(best, best);
            int32_t stack[kStackSize];
            float kstack[kStackSize];
            int sp = 0;
            int32_t cur = sc.root_is_leaf ? pack_leaf(0, sc.num_tris) : 0;
            for (;;) {
                if (cur >= 0) {
                    if (COUNT) visits++;
                    const float kOut = __int_as_float(0x7f800000);  // +inf: a pruned child
                    if (WIDE) {
                        uint32_t a[8], b[8];
                        ldg256u(sc.nodes4 + 4 * cur, a);
                        ldg256u(sc.nodes4 + 4 * cur + 2, b);
                        // unused slots carry a degenerate box and triangle 0's leaf: visiting one re-tests a triangle
                        int32_t c[4] = {(int32_t)b[4], (int32_t)b[5], (int32_t)b[6], (int32_t)b[7]};
                        float t[4];
                        t[0] = box_bound2(a[0], a[1], a[2], g);
                        t[1] = box_bound2(a[3], a[4], a[5], g);
                        t[2] = box_bound2(a[6], a[7], b[0], g);
                        t[3] = box_bound2(b[1], b[2], b[3], g);
                        // kept children at most FLT_MAX, pruned ones +inf, so the sort below leaves pruned ones last
#pragma unroll
                        for (int k = 0; k < 4; k++) t[k] = t[k] <= bestSq ? fminf(t[k], 3.4028235e38f) : kOut;
#define RT_CE(i, j)                                   \
    {                                                 \
        const bool sw = t[j] < t[i];                  \
        const float lo = fminf(t[i], t[j]);           \
        const float hi = fmaxf(t[i], t[j]);           \
        const int32_t ci = sw ? c[j] : c[i];          \
        const int32_t cj = sw ? c[i] : c[j];          \
        t[i] = lo; t[j] = hi; c[i] = ci; c[j] = cj;   \
    }
                        RT_CE(0, 1) RT_CE(2, 3) RT_CE(0, 2) RT_CE(1, 3) RT_CE(1, 2)
#undef RT_CE
                        if (t[3] < kOut) { stack[sp] = c[3]; kstack[sp] = t[3]; sp++; }
                        if (t[2] < kOut) { stack[sp] = c[2]; kstack[sp] = t[2]; sp++; }
                        if (t[1] < kOut) { stack[sp] = c[1]; kstack[sp] = t[1]; sp++; }
                        if (t[0] < kOut) { cur = c[0]; continue; }
                    } else {
                        uint32_t w[8];
                        ldg256u(sc.nodes + 2 * cur, w);
                        const float l = box_bound2(w[0], w[1], w[2], g);
                        const float rr = box_bound2(w[3], w[4], w[5], g);
                        const bool hitL = l <= bestSq, hitR = rr <= bestSq;
                        const int32_t cl = (int32_t)w[6], cr = (int32_t)w[7];
                        if (hitL && hitR) {
                            const bool leftFirst = l <= rr;
                            stack[sp] = leftFirst ? cr : cl;
                            kstack[sp] = leftFirst ? rr : l;
                            sp++;
                            cur = leftFirst ? cl : cr;
                            continue;
                        }
                        if (hitL || hitR) {
                            cur = hitL ? cl : cr;
                            continue;
                        }
                    }
                } else {
                    const int32_t packed = ~cur;
                    const int32_t first = packed & kLeafFirstMask;
                    const int32_t count = (packed >> kLeafCountShift) + 1;
                    for (int32_t s = first; s < first + count; s++) {
                        V3 a, e0, e1;
                        load_tri36(sc, s, a, e0, e1);
                        if (COUNT) tests++;
                        float u, v;
                        const float d = point_triangle(p, a, e0, e1, u, v);
                        bool take = d < best;
                        if (!take && d == best) {  // exact tie: the lower original id wins
                            const int32_t o = __ldg(&sc.tri_orig[s]);
                            if (bestSlot >= 0 && bestOrig < 0) bestOrig = __ldg(&sc.tri_orig[bestSlot]);
                            take = bestSlot < 0 || o < bestOrig;
                            if (take) bestOrig = o;
                        } else if (take) {
                            bestOrig = -1;
                        }
                        if (take) {
                            if (d < best) bestSq = __fmul_ru(d, d);
                            best = d;
                            bu = u;
                            bv = v;
                            bestSlot = s;
                        }
                    }
                }
                // pop the nearest pending subtree that can still hold a distance <= best
                bool got = false;
                while (sp > 0) {
                    --sp;
                    if (kstack[sp] <= bestSq) {
                        cur = stack[sp];
                        got = true;
                        break;
                    }
                }
                if (!got) break;
            }
        }
        const bool hit = bestSlot >= 0;
        if (qa.tri) qa.tri[i] = hit ? (bestOrig >= 0 ? bestOrig : __ldg(&sc.tri_orig[bestSlot])) : -1;
        if (qa.dist) qa.dist[i] = hit ? best : kMissT;
        if (qa.bu) qa.bu[i] = hit ? bu : 0.0f;
        if (qa.bv) qa.bv[i] = hit ? bv : 0.0f;
        if (qa.closest) {
            V3 pt = v3(0.0f, 0.0f, 0.0f);
            if (hit) {
                V3 a, e0, e1;
                load_tri36(sc, bestSlot, a, e0, e1);
                pt = a + (e0 * bu + e1 * bv);
            }
            qa.closest[3 * i] = pt.x;
            qa.closest[3 * i + 1] = pt.y;
            qa.closest[3 * i + 2] = pt.z;
        }
    }
    if (COUNT) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            visits += __shfl_xor_sync(0xffffffffu, visits, off);
            tests += __shfl_xor_sync(0xffffffffu, tests, off);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&stats[2], (unsigned long long)visits);
            atomicAdd(&stats[3], (unsigned long long)tests);
        }
    }
}

cudaError_t wf_nearest(const Launcher& L, const SceneView& sc, const NearestArgs& q, int64_t n,
                       unsigned long long* stats) {
    if (n <= 0) return cudaSuccess;
    const int blocks = (int)((n + kNearBlock - 1) / kNearBlock);
    const bool wide = sc.nodes4 != nullptr;
#define RT_NEAR(C, W) k_nearest<C, W><<<blocks, kNearBlock, 0, L.st>>>(sc, q, (long long)n, stats)
    if (wide) { if (L.instrument) RT_NEAR(true, true); else RT_NEAR(false, true); }
    else { if (L.instrument) RT_NEAR(true, false); else RT_NEAR(false, false); }
#undef RT_NEAR
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

}  // namespace rt
