// nearest_oracle.cpp — CPU reference of the nearest-triangle query (rt_query_nearest).  TEST INFRASTRUCTURE ONLY:
// tests/nearest_oracle.py loads it; nothing under raytracing2-fork_b200/ includes, links or calls it.
//
// Build with -ffp-contract=off, like the oracle: every expression is evaluated in binary32 in exactly the order
// written, the order raytracing2-fork_b200/csrc/nearest.cu (compiled with -fmad=false) follows, so the two agree
// bit for bit (DESIGN.md §4, §5).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <thread>
#include <vector>

#include "../../include/rt_b200.h"

namespace {

struct V3 {
    float x, y, z;
};
inline V3 v3(float x, float y, float z) { return V3{x, y, z}; }
inline V3 v3(const float* p) { return V3{p[0], p[1], p[2]}; }
inline V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
// dot3 = (a.x*b.x + a.y*b.y) + a.z*b.z, the order of glm and of rt_math.cuh
inline float dot(V3 a, V3 b) {
    const float tx = a.x * b.x, ty = a.y * b.y, tz = a.z * b.z;
    return (tx + ty) + tz;
}

// Distance from p to the closed triangle (a, e0 = b - a, e1 = c - a): the definition k_nearest (csrc/nearest.cu
// nearest_uv / point_triangle) reproduces bit for bit.  e0 and e1 are computed exactly as the GPU's triangle records
// store them (bvh_build.cu: e0 = b - a, e1 = c - a); recomputing b or c from a would round differently.
// Ericson, Real-Time Collision Detection §5.1.5, restated on (a, e0, e1), every operation in this order:
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
// An edge case is taken only when its denominator is > 0 and its quotient <= 1 (no 0 / 0, no inf / inf); otherwise
// the tests go on, and degenerate triangles end in the segment fallback, which never divides by zero.
inline float clamp01(float x) {
    x = x > 0.0f ? x : 0.0f;  // NaN -> 0
    return x < 1.0f ? x : 1.0f;
}
void nearestUV(V3 ap, V3 e0, V3 e1, float& u, float& v) {
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
// dist, (u, v) and the closest point a + q
float pointTriangle(V3 p, const rt_triangle& t, float& u, float& v, V3& point) {
    const V3 a = v3(t.a), b = v3(t.b), c = v3(t.c);
    const V3 e0 = b - a, e1 = c - a;
    const V3 ap = p - a;
    nearestUV(ap, e0, e1, u, v);
    const V3 q = e0 * u + e1 * v;
    const V3 d = ap - q;
    point = a + q;
    return sqrtf(dot(d, d));
}

}  // namespace

extern "C" {

float nro_point_triangle(const float p[3], const rt_triangle* t, float* u, float* v, float closest[3]) {
    float uu = 0.0f, vv = 0.0f;
    V3 pt;
    const float d = pointTriangle(v3(p), *t, uu, vv, pt);
    if (u) *u = uu;
    if (v) *v = vv;
    if (closest) {
        closest[0] = pt.x;
        closest[1] = pt.y;
        closest[2] = pt.z;
    }
    return d;
}

// Brute force over every triangle of the caller's array: for each point and radius r (max_dist NULL = unbounded), the
// smallest dist(p, T) < min(r, 1e38), exact ties to the lowest index; a NaN, zero or negative r and a point with a
// non-finite coordinate miss.  A miss writes -1 / 1e38 / 0 / 0 and (0, 0, 0).  Outputs may be NULL.
int nro_nearest_points(const rt_triangle* tris, int64_t n, const float* points, const float* max_dist, int64_t count,
                       int32_t* tri_id, float* dist, float* bu, float* bv, float* closest) {
    if (n < 0 || count < 0 || (n > 0 && !tris) || (count > 0 && !points)) return RT_ERR_INVALID;
    auto one = [&](int64_t i) {
        const V3 p = v3(points + 3 * i);
        const float r = max_dist ? max_dist[i] : 1e38f;
        const float limit = r < 1e38f ? r : 1e38f;
        int32_t bestId = -1;
        float best = 1e38f, bestU = 0.0f, bestV = 0.0f;
        V3 bestP = v3(0.0f, 0.0f, 0.0f);
        if (r > 0.0f && std::isfinite(p.x) && std::isfinite(p.y) && std::isfinite(p.z)) {
            for (int64_t k = 0; k < n; k++) {
                float u, v;
                V3 pt;
                const float d = pointTriangle(p, tris[k], u, v, pt);
                if (d < limit && (bestId < 0 || d < best)) {  // k ascends: an exact tie keeps the lower index
                    best = d; bestU = u; bestV = v; bestP = pt; bestId = (int32_t)k;
                }
            }
        }
        if (tri_id) tri_id[i] = bestId;
        if (dist) dist[i] = bestId >= 0 ? best : 1e38f;
        if (bu) bu[i] = bestU;
        if (bv) bv[i] = bestV;
        if (closest) {
            closest[3 * i] = bestP.x;
            closest[3 * i + 1] = bestP.y;
            closest[3 * i + 2] = bestP.z;
        }
    };
    const int threads = std::max(1, (int)std::thread::hardware_concurrency());
    std::atomic<int64_t> next(0);
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; t++)
        pool.emplace_back([&]() {
            for (;;) {
                const int64_t i0 = next.fetch_add(256);
                if (i0 >= count) break;
                for (int64_t i = i0; i < std::min(count, i0 + 256); i++) one(i);
            }
        });
    for (auto& th : pool) th.join();
    return RT_OK;
}

}  // extern "C"
