// wavefront.cu — the per-pixel hot path as wavefront kernels (replaces the megakernel
// RayTracing/Assets/Shaders/compute.glsl; citations S:line refer to that file, R:line to
// RayTracing/src/rayTracing.cpp).
//
//   k_seed_pixels   S:668       per-pixel seed of the reference's sequential stream (PCG mode)
//   k_raygen        S:660-690   NDC of the pixel corner, defocus arc, +-1/4 pixel jitter, first ray
//   k_extend        S:410-460   closest hit of every live path: persistent warps over the 4-wide tree
//                               (node_step4) or the binary one (node_step), slab tests in rt_scene.cuh
//   k_shade         S:472-563   one bounce: material switch, next ray, Russian roulette; survivors
//                               are compacted into the next queue with warp ballot + prefix popcount
//   k_accumulate    S:692       per-pixel sum of the batch's samples, in sample order
//   k_resolve       S:696-700   mean, ACES, gamma, image store; + unorm8 quantise and add (R:194-238)
//   k_finalize      R:248-259   average of the 8-bit frames, truncate, flip
//   k_preview       S:565-645   traceBasic, one thread per pixel (interactive preview)
//   k_first_rays                the camera rays of the first-hit parity hook, traced by k_extend's CLOSEST query
//
// A "path slot" is (lane, pixel): a batch holds frames_in_batch x samples_in_batch lanes of every pixel
// (FrameParams, rt_internal.h) and each slot owns one float4 of `contrib`; the radiance of a path is a single value written at its
// terminal event (light hit / miss / error colour), so k_accumulate can add the lanes in sample
// order and the image does not depend on the order in which paths finish.
#include <type_traits>

#include "rt_internal.h"

namespace rt {

constexpr int kBlock = 256;

struct Material {
    V3 color, emission;
    int32_t textureIndex;
    float emissionStrength, smoothness, specularProbability, checkerScale, refractiveIndex;
    int32_t type, isEdgeHighlight;
};
__device__ __forceinline__ Material load_material(const SceneView& sc, int32_t idx) {
    const float4 m0 = __ldg(&sc.materials[6 * idx + 0]);
    const float4 m2 = __ldg(&sc.materials[6 * idx + 2]);
    const float4 m3 = __ldg(&sc.materials[6 * idx + 3]);
    const float4 m4 = __ldg(&sc.materials[6 * idx + 4]);
    const float4 m5 = __ldg(&sc.materials[6 * idx + 5]);
    Material m;
    m.color = v3(m0);
    m.emission = v3(m2);
    m.textureIndex = __float_as_int(m3.x);
    m.emissionStrength = m3.y;
    m.smoothness = m3.z;
    m.specularProbability = m3.w;
    m.checkerScale = m4.x;
    m.refractiveIndex = m4.y;
    m.type = __float_as_int(m4.z);
    m.isEdgeHighlight = __float_as_int(m5.x);
    return m;
}

// GL_LINEAR / GL_REPEAT / unorm8, no mips (external/OpenGL/textureClass.cpp:95-101); DESIGN.md §4.6
// b / 255.0f for a byte, bit for bit, without the IEEE division sequence: one Newton correction of the product with
// the rounded reciprocal is the correctly rounded quotient for every b in 0..255 (checked exhaustively with exact
// rationals, tests/test_oracle_cpu.py::test_unorm8_reciprocal_sequence_is_exact; the plain product is wrong for 126).
__device__ __forceinline__ float unorm8(uint8_t b) {
    const float x = (float)b;
    const float c = 0.003921568859368563f;  // RN(1 / 255)
    const float q0 = __fmul_rn(x, c);
    const float r = __fmaf_rn(-255.0f, q0, x);
    return __fmaf_rn(r, c, q0);
}
__device__ __forceinline__ V3 texel(const uint8_t* __restrict__ px, int w, int ch, int i, int j) {
    const uint8_t* p = px + ((size_t)j * w + i) * ch;
    const float r = unorm8(__ldg(p));
    if (ch == 1) return v3(r, r, r);
    const float g = unorm8(__ldg(p + 1));
    if (ch == 2) return v3(r, g, 0.0f);
    return v3(r, g, unorm8(__ldg(p + 2)));
}
__device__ __forceinline__ V3 sample_texture(const SceneView& sc, int t, float u, float v) {
    const int w = sc.tex_w[t], h = sc.tex_h[t], ch = sc.tex_ch[t];
    if (w <= 0 || h <= 0) return v3(0.0f, 0.0f, 0.0f);
    float s = u - floorf(u);
    float r = v - floorf(v);
    if (!(s >= 0.0f && s <= 1.0f)) s = 0.0f;
    if (!(r >= 0.0f && r <= 1.0f)) r = 0.0f;
    const float fx = s * (float)w - 0.5f;
    const float fy = r * (float)h - 0.5f;
    const float flx = floorf(fx), fly = floorf(fy);
    const float ax = fx - flx, ay = fy - fly;
    // REPEAT: s, r in [0, 1] put floor(fx) in [-1, w-1] and its right neighbour in [0, w], so the positive modulo
    // ((i % w) + w) % w of the specification is one conditional add / subtract (eight integer divisions saved)
    int i0 = (int)flx, j0 = (int)fly;
    int i1 = i0 + 1, j1 = j0 + 1;
    i0 = i0 < 0 ? i0 + w : i0;
    j0 = j0 < 0 ? j0 + h : j0;
    i1 = i1 >= w ? i1 - w : i1;
    j1 = j1 >= h ? j1 - h : j1;
    const uint8_t* px = sc.tex_px[t];
    const float w00 = (1.0f - ax) * (1.0f - ay), w10 = ax * (1.0f - ay), w01 = (1.0f - ax) * ay, w11 = ax * ay;
    return ((texel(px, w, ch, i0, j0) * w00 + texel(px, w, ch, i1, j0) * w10) + texel(px, w, ch, i0, j1) * w01) +
           texel(px, w, ch, i1, j1) * w11;
}
// S:342-368
__device__ __forceinline__ V3 triangle_texture_color(const SceneView& sc, int numTextures, int textureIndex,
                                                     float bw, float bu, float bv, int32_t slot) {
    const float4 s0 = __ldg(&sc.tri_shade[2 * slot + 0]);
    const float4 s1 = __ldg(&sc.tri_shade[2 * slot + 1]);
    const float uvx = (s0.x * bu + s0.z * bv) + s1.x * bw;
    const float uvy = (s0.y * bu + s0.w * bv) + s1.y * bw;
    if (textureIndex < 0 || textureIndex >= numTextures) return v3(0.0f, 0.0f, 0.0f);
    if (textureIndex >= RT_MAX_TEXTURES) return v3(1.0f, 0.0f, 1.0f);
    return sample_texture(sc, textureIndex, uvx, uvy);
}

// S:216-273
__device__ __noinline__ V3 env_light(V3 dir) {
    const V3 sunDir = normalize(v3(0.6f, 0.3f, -0.2f));
    const float sunDot = dot(dir, sunDir);
    const float horizonDot = dir.y;
    const V3 zenithColor = v3(0.15f, 0.25f, 0.65f), deepOrange = v3(1.2f, 0.4f, 0.1f),
             yellow = v3(1.0f, 0.8f, 0.3f), coolBlue = v3(0.3f, 0.4f, 0.7f), groundColor = v3(0.2f, 0.15f, 0.1f);
    const float sunToOpposite = (dot(dir, -sunDir) + 1.0f) * 0.5f;
    V3 horizonColor;
    if (sunToOpposite < 0.5f)
        horizonColor = mix(deepOrange, yellow, sunToOpposite * 2.0f);
    else
        horizonColor = mix(yellow, coolBlue, (sunToOpposite - 0.5f) * 2.0f);
    const float skyGradient = smoothstep(-0.2f, 0.8f, horizonDot);
    const V3 baseColor = mix(horizonColor, zenithColor, skyGradient);
    const V3 sunCenter = v3(15.0f, 15.0f, 10.0f);
    const float sunAngle = acos_(gclamp(sunDot, -1.0f, 1.0f));
    const float glow1 = exp_(-sunAngle * 600.0f);
    const float glow2 = exp_(-sunAngle * 150.0f) * 0.3f;
    const float glow3 = exp_(-sunAngle * 60.0f) * 0.1f;
    const float glow4 = exp_(-sunAngle * 15.0f) * 0.03f;
    const float totalGlow = ((glow1 + glow2) + glow3) + glow4;
    V3 finalColor = baseColor + sunCenter * totalGlow;
    if (horizonDot < 0.0f) {
        const float groundBlend = smoothstep(-0.1f, 0.0f, horizonDot);
        finalColor = mix(groundColor, finalColor, groundBlend);
        const float groundSunGlow = exp_(-sunAngle * 15.0f) * 0.2f;
        finalColor = finalColor + (sunCenter * groundSunGlow) * 0.05f;
    }
    return finalColor;
}

// S:201-214
__device__ __forceinline__ V3 refract_(V3 I, V3 N, float eta, bool& isRefracted) {
    const float k = 1.0f - eta * eta * (1.0f - dot(N, I) * dot(N, I));
    if (k < 0.0f) {
        isRefracted = false;
        return reflect(I, N);
    }
    isRefracted = true;
    return I * eta - N * (eta * dot(N, I) + sqrtf(k));
}
__device__ __forceinline__ bool black_checker(V3 p, float scale) {  // S:524-527
    if (!(scale > 0.0f)) return false;
    const float sum = (floorf(p.x * scale) + floorf(p.y * scale)) + floorf(p.z * scale);
    const float m = sum - 2.0f * floorf(sum / 2.0f);
    return m == 0.0f;
}
// normalize(cross(e0, e1)) of S:331, evaluated once per triangle by k_emit_tris with the same operations
__device__ __forceinline__ V3 tri_normal(const SceneView& sc, int32_t slot) {
    const float4 g3 = __ldg(&sc.tri_geom[4 * slot + 3]);
    return v3(g3.x, g3.y, g3.z);
}

// pixel geometry shared by raygen / first-hit / preview (S:663-676)
struct PixelSetup {
    V3 endPoint, centreDir;
    uint32_t seed, pixelId;
};
__device__ __forceinline__ PixelSetup pixel_setup(const rt_uniforms& u, int tx, int ty) {
    const int W = (int)u.width, H = (int)u.height;
    const float x = (float)(tx * 2 - W) / (float)W;
    const float y = (float)(ty * 2 - H) / (float)H;
    PixelSetup ps;
    ps.pixelId = (uint32_t)tx + (uint32_t)ty * (uint32_t)W;
    ps.seed = ps.pixelId + u.frameIndex * 968824447u;
    const V3 cam = v3(u.cameraPos), vf = v3(u.viewportFront), vr = v3(u.viewportRight), vu = v3(u.viewportUp);
    ps.endPoint = ((cam + vf) + vr * x) + vu * y;
    ps.centreDir = normalize((vf + vr * x) + vu * y);
    return ps;
}
template <class R>
__device__ __forceinline__ void sample_ray(const rt_uniforms& u, const PixelSetup& ps, R& rng, V3& o, V3& d) {
    const float angle = rng.next();  // S:163
    const float cx = cos01(angle), sy = sin01(angle);
    o = (v3(u.cameraPos) + v3(u.defocusDiskRight) * cx) + v3(u.defocusDiskUp) * sy;
    const float jr = -0.5f + (0.5f - -0.5f) * rng.next();  // random(-0.5, 0.5, seed), S:156-159
    const float ju = -0.5f + (0.5f - -0.5f) * rng.next();
    const V3 endJ = (ps.endPoint + v3(u.pixelRight) * jr) + v3(u.pixelUp) * ju;
    d = normalize(endJ - o);
}
__device__ __forceinline__ void local_pixel_xy(const FrameParams& fp, int p, int& tx, int& ty) {
    const int r = (int)fastdiv((uint32_t)p, fp.div_width);
    tx = p - r * fp.width;
    ty = fp.rows ? fp.rows[r] : r;
}
// tx + ty * W of a local pixel; without a row table (no tile split) that is the local index itself
__device__ __forceinline__ uint32_t local_pixel_id(const FrameParams& fp, int p) {
    if (!fp.rows) return (uint32_t)p;
    int tx, ty;
    local_pixel_xy(fp, p, tx, ty);
    return (uint32_t)tx + (uint32_t)ty * fp.u.width;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_seed_pixels(const __grid_constant__ FrameParams fp,
                                                        uint32_t* __restrict__ pix_rng) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= fp.local_pixels * fp.frames_in_batch) return;
    const int k = i / fp.local_pixels;
    const int p = i - k * fp.local_pixels;
    int tx, ty;
    local_pixel_xy(fp, p, tx, ty);
    const uint32_t frame = fp.u.frameIndex + (uint32_t)(k * fp.frame_stride);
    pix_rng[i] = (uint32_t)tx + (uint32_t)ty * fp.u.width + frame * 968824447u;  // S:668
}

__global__ void __launch_bounds__(kBlock) k_clear_accum(float4* __restrict__ accum, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) accum[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

template <int MODE>
__global__ void __launch_bounds__(kBlock) k_raygen(const __grid_constant__ FrameParams fp, PathArrays cur,
                                                   float4* __restrict__ contrib, uint32_t* __restrict__ pix_rng,
                                                   uint32_t* __restrict__ counts, int ncounts,
                                                   unsigned long long* __restrict__ stats) {
    const int n = fp.local_pixels * fp.lanes_active;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        counts[0] = (uint32_t)n;
        for (int k = 1; k < 2 * ncounts; k++) counts[k] = 0u;  // live counts, then the extend cursors
        atomicAdd(&stats[1], (unsigned long long)n);
    }
    if (i >= n) return;
    const int lane = i / fp.local_pixels;
    const int p = i - lane * fp.local_pixels;
    int tx, ty;
    local_pixel_xy(fp, p, tx, ty);
    const PixelSetup ps = pixel_setup(fp.u, tx, ty);
    const int k = lane / fp.samples_in_batch;  // batch frame
    const int s = lane - k * fp.samples_in_batch;
    const uint32_t frame = fp.u.frameIndex + (uint32_t)(k * fp.frame_stride);
    Rng<MODE> rng;
    rng.init(MODE == 0 ? pix_rng[(size_t)k * fp.local_pixels + p] : (uint32_t)(fp.sample_base + s), ps.pixelId, frame, 0u);
    rng.stream(0u);
    V3 o, d;
    sample_ray(fp.u, ps, rng, o, d);
    cur.od0[i] = make_float4(o.x, o.y, o.z, d.x);
    cur.od1[i] = make_float4(d.y, d.z, 1.0f, 1.0f);
    cur.misc[i] = make_float4(1.0f, __int_as_float(i), __uint_as_float(rng.carry()), __int_as_float(0));
    // every path writes its slot of `contrib` exactly once, at its terminal event in k_shade (the bounce limit is
    // one); only a frame without any bounce needs the zero
    if (fp.u.maxBounceCount <= 0 || fp.debug_zero_contrib) contrib[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

// ---------------------------------------------------------------------------------------------- k_extend
// Persistent warps.  Every lane owns at most one ray; finished lanes are refilled from the queue
// through a device-side cursor (one atomicAdd per refill, claimed by the first idle lane), so a warp
// never waits for its slowest ray.  Each iteration the warp VOTES on what to execute: a leaf step
// (exact Möller–Trumbore, compute.glsl:302-340) when at least `leafVote` lanes are parked at a leaf or
// nobody can take a node step, otherwise a few node steps (two or four slab tests each) — both are executed under a
// warp-uniform branch, so the instruction stream never serialises node and triangle code inside one
// iteration.  ncu on the v1 kernel (one thread per ray, per-lane if/else) showed 6.85 of 32 lanes
// active per instruction; this structure is what that measurement asked for
// (profiles/r1_v1_extend_ncu_full.md).
//
// The closest-hit rule (min dst, then lowest original index) makes the result independent of the
// order in which lanes, nodes and triangles are visited, so the restructuring changes no bit.
constexpr int kExtBlock = 128;
constexpr int kExtMinBlocks = 9;  // 56 registers: nine resident blocks per SM (ten at 48 registers measured 0.8 % slower, eight slower too)
// Rays claimed from the queue per atomicAdd on the shared cursor.  Round 1 took one atomic per refill.
constexpr uint32_t kExtClaim = 128;
// Software prefetch of the streaming ray records.  With chunked claims the warp knows its next records exactly, and
// at every refill it prefetches the head of its private range into L2.  Measured and not kept: the same into L1, the
// whole chunk that some warp will claim one generation ahead (it is evicted again before it is used often enough to
// cost 8 B of DRAM traffic per segment: ncu, profiles/r2_traffic_*.csv of the v20 capture), and no prefetch.  Before
// chunked claims, prefetching the record a lane would claim one refill generation later gave
// config 2 5859 vs 5806 Mrays/s (+0.9 %; profiles/r2_prefetch_ab.txt).
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
constexpr int32_t kPop = (int32_t)0x80000000;       // lane state: take the next subtree from the stack
constexpr int32_t kIdle = (int32_t)0x80000001;      // lane state: no ray
// Warp-vote thresholds: a leaf step when >= kLeafVote lanes wait at a leaf, a refill when >= kRefill lanes are idle.
// Refill 4 / 6 / 12 and leaf vote 12 / 16 measured 0.2-1.7 % slower (DESIGN.md section 5).
constexpr int kLeafVote = 14;
constexpr int kRefill = 8;

// One node step for a lane at an inner node: two slab tests, then a branch-free choice of the next
// state (near child / push far child / pop).  v2's if/else ladder here ran at 3-8 active lanes
// (profiles/r1_v2_extend_ncu_full.md); selects and one predicated store keep the warp converged.
struct RayRegs {
    V3 o, d;      // world space: the exact triangle test
    GridRay g;    // grid space: the slab tests
    float bestT;
};
// Traversal stack: the first kShStack entries of every lane live in shared memory laid out
// [level][thread], so a warp-wide push or pop is conflict-free (one bank pair per lane) whatever
// the lanes' depths are; in local memory the same access scatters over up to 32 lines and costs up
// to 32 L1TEX wavefronts.  Deeper entries (rare: most rays keep fewer than 16 pending nodes) overflow to local memory.
constexpr int kShStack = 16;
struct Stack {
    int2* sh;         // &shared[0][threadIdx.x]; stride kExtBlock
    int32_t* ovNode;  // local overflow
    float* ovT;
    __device__ __forceinline__ void push(int sp, int32_t c, float t) {
        if (sp < kShStack) sh[sp * kExtBlock] = make_int2(c, __float_as_int(t));
        else { ovNode[sp - kShStack] = c; ovT[sp - kShStack] = t; }
    }
    __device__ __forceinline__ void get(int sp, int32_t& c, float& t) const {
        if (sp < kShStack) { const int2 e = sh[sp * kExtBlock]; c = e.x; t = __int_as_float(e.y); }
        else { c = ovNode[sp - kShStack]; t = ovT[sp - kShStack]; }
    }
    // DEEP = false: the caller guarantees sp < kShStack (shared entries only, no overflow code at all)
    template <bool DEEP>
    __device__ __forceinline__ void pushT(int sp, int32_t c, float t) {
        if (DEEP) push(sp, c, t);
        else sh[sp * kExtBlock] = make_int2(c, __float_as_int(t));
    }
    template <bool DEEP>
    __device__ __forceinline__ void getT(int sp, int32_t& c, float& t) const {
        if (DEEP) { get(sp, c, t); }
        else { const int2 e = sh[sp * kExtBlock]; c = e.x; t = __int_as_float(e.y); }
    }
};
template <bool DEEP, bool WIDEN>
__device__ __forceinline__ void node_step(const SceneView& sc, const RayRegs& r, int32_t& node, int& sp, Stack& st) {
    uint32_t w[8];
    ldg256u(sc.nodes + 2 * node, w);
    float lNear, rNear;
    bool hitL, hitR;
    slab2<WIDEN>(w, r.g, r.bestT, lNear, rNear, hitL, hitR);
    const int32_t cl = (int32_t)w[6], cr = (int32_t)w[7];
    // a missed child is infinitely far: the near / far choice, "both" and "any" then come out of one compare,
    // one min and one max instead of a predicate ladder
    const float kFar = 3.0e38f;
    const float lN = hitL ? lNear : kFar, rN = hitR ? rNear : kFar;
    const bool goLeft = lN <= rN;
    const float farT = fmaxf(lN, rN);
    const bool both = farT < kFar;
    const bool any = fminf(lN, rN) < kFar;
    if (both) st.pushT<DEEP>(sp, goLeft ? cr : cl, farT);
    sp += both ? 1 : 0;
    node = any ? (goLeft ? cl : cr) : kPop;
}

// The same step over a 4-wide node (64 bytes, two 256-bit loads): four slab tests, a 5-comparator sorting network
// on (entry distance, child) with missed children at +inf, the nearest child becomes the lane's node and the other
// hit children are pushed farthest first.  Up to three pushes per step.
// (Staging the root and the three levels below it in shared memory measured -3 %: those nodes are L1 hits already.)
template <bool DEEP, bool WIDEN>
__device__ __forceinline__ void node_step4(const SceneView& sc, const RayRegs& r, int32_t& node, int& sp, Stack& st) {
    uint32_t a[8], b[8];
    ldg256u(sc.nodes4 + 4 * node, a);
    ldg256u(sc.nodes4 + 4 * node + 2, b);
    float t[4];
    int32_t c[4] = {(int32_t)b[4], (int32_t)b[5], (int32_t)b[6], (int32_t)b[7]};
    t[0] = slab1<WIDEN>(a[0], a[1], a[2], r.g, r.bestT);
    t[1] = slab1<WIDEN>(a[3], a[4], a[5], r.g, r.bestT);
    t[2] = slab1<WIDEN>(a[6], a[7], b[0], r.g, r.bestT);
    t[3] = slab1<WIDEN>(b[1], b[2], b[3], r.g, r.bestT);
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
    if (t[3] < kSlabMiss) { st.pushT<DEEP>(sp, c[3], t[3]); sp++; }
    if (t[2] < kSlabMiss) { st.pushT<DEEP>(sp, c[2], t[2]); sp++; }
    if (t[1] < kSlabMiss) { st.pushT<DEEP>(sp, c[1], t[1]); sp++; }
    node = t[0] < kSlabMiss ? c[0] : kPop;
}

constexpr int32_t kDrain = (int32_t)0x80000002;     // lane state (SPEC): stack empty, a postponed leaf still to test
constexpr int32_t kNoLeaf = (int32_t)0x80000003;    // `post` holds no leaf
__device__ __forceinline__ bool is_leaf_code(int32_t x) { return x < 0 && (uint32_t)x > (uint32_t)kNoLeaf; }

// SPEC = speculative traversal (Aila & Laine's "postponed leaf"): a lane that reaches a leaf parks it in
// `post` and keeps descending; it only has to wait for a leaf step when it reaches a SECOND leaf (or runs
// out of nodes).  Node steps then run with more lanes, leaf steps test up to two leaves per lane; the price
// is a stale bestT while a leaf is parked (a few more node visits).  How far a lane runs ahead of its parked leaf
// depends on the other lanes of its warp, so the instrumented variants (COUNT) walk without it: their node-visit
// and triangle-test counts are those of each ray's own sequential walk.
//
// Q = CLOSEST / ANY serve the ray queries: the refill reads the caller's (N, 3) arrays and an optional tmax, the pop
// phase writes the caller's outputs, and everything they add sits behind `if constexpr`, so the RENDER instantiations
// compile as before (`qa` is appended to the parameters and never read by them).  The hit rule of a query: a triangle
// counts iff 1e-6 < dst < min(tmax, kMissT).  bestT starts at the largest float below that bound, which turns the
// traversal's `dst <= bestT` into `dst < bound` (DESIGN.md, "Ray queries").
template <bool COUNT, bool WIDE, bool WIDEN, Query Q>
__global__ void __launch_bounds__(kExtBlock, kExtMinBlocks) k_extend(const __grid_constant__ SceneView sc, PathArrays cur,
                                                      float4* __restrict__ hit, const uint32_t* __restrict__ count,
                                                      uint32_t* __restrict__ cursor,
                                                      unsigned long long* __restrict__ stats,
                                                      const __grid_constant__ QueryArgs qa) {
    constexpr bool SPEC = !COUNT;
    constexpr bool ANY = Q == Query::ANY;
    constexpr int kNodeSteps = WIDE ? 2 : 4;  // node steps per vote (3 on the 4-wide tree, 3 / 6 on the binary one: slower)
    const uint32_t n = *count;
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)n);
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t ltMask = (1u << lane) - 1u;
    constexpr uint32_t FULL = 0xffffffffu;
    const float kWiden = WIDEN ? kWidenFar : 1.0f;  // x * 1.0f folds away

    __shared__ int2 shStack[kShStack][kExtBlock];
    __shared__ uint32_t sClaim[kExtBlock / 32][4];  // per warp: next, end of its private range; queue exhausted
    if ((threadIdx.x & 31u) == 0u) { sClaim[threadIdx.x >> 5][0] = 0u; sClaim[threadIdx.x >> 5][1] = 0u; sClaim[threadIdx.x >> 5][2] = 0u; }
    __syncwarp();
    int32_t ovNode[kStackSize - kShStack];
    float ovT[kStackSize - kShStack];
    Stack st{&shStack[0][threadIdx.x], ovNode, ovT};
    bool exhausted = (n == 0u) || sc.num_tris <= 0;
    uint32_t ray = 0;
    RayRegs r;
    r.o = v3(0, 0, 0); r.d = v3(0, 0, 1); r.bestT = kMissT;
    r.g.ox = r.g.oy = r.g.oz = r.g.ix = r.g.iy = r.g.iz = r.g.nx = r.g.ny = r.g.nz = 0.0f;
    float bestU = 0, bestV = 0;
    int32_t bestSlot = -1;
    int32_t node = kIdle;
    int32_t post = kNoLeaf;
    int sp = 0;
    uint32_t visits = 0, tests = 0;

    // the result of ray `i` (a query writes the caller's arrays; a miss is -1 / kMissT / 0 / 0, or "not occluded")
    auto write_result = [&](uint32_t i) {
        if constexpr (Q == Query::RENDER) {
            hit[i] = make_float4(r.bestT, bestU, bestV, __int_as_float(bestSlot));
        } else if constexpr (ANY) {
            qa.occluded[i] = bestSlot >= 0 ? 1 : 0;
        } else {
            const bool h = bestSlot >= 0;
            if (qa.tri) qa.tri[i] = h ? __ldg(&sc.tri_orig[bestSlot]) : -1;
            if (qa.dst) qa.dst[i] = h ? r.bestT : kMissT;
            if (qa.bu) qa.bu[i] = h ? bestU : 0.0f;
            if (qa.bv) qa.bv[i] = h ? bestV : 0.0f;
        }
    };
    if (sc.num_tris <= 0) {  // empty scene: every ray misses
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            if constexpr (Q == Query::RENDER) hit[i] = make_float4(kMissT, 0.0f, 0.0f, __int_as_float(-1));
            else write_result(i);
        }
    }

    // exact Möller–Trumbore against every triangle of one leaf; min (dst, original index) wins
    auto test_tri = [&](int32_t s) {
        const TriGeom tg = load_tri(sc, s);
        if (COUNT) tests++;
        float dst, u, v;
        // the test leaves before the barycentrics when dst > best
        if (ray_triangle(r.o, r.d, tg.a, tg.e0, tg.e1, tg.N, dst, u, v, r.bestT)) {
            // the original indices are needed only to break an exact tie in dst: fetch them then, not for every
            // candidate (the dependent 4-byte gather was 3.4 % of k_extend's stall samples)
            if (dst <= r.bestT && dst < kMissT) {
                bool take = dst < r.bestT;
                if constexpr (Q == Query::RENDER) {
                    if (!take) take = __ldg(&sc.tri_orig[s]) < __ldg(&sc.tri_orig[bestSlot]);  // bestT < kMissT: bestSlot >= 0
                } else if constexpr (ANY) {
                    take = true;  // any accepted triangle answers the query
                } else {
                    // a query's bestT starts at the bound itself (dst == bestT is a hit), so the first candidate
                    // must be taken without the tie-break: there is no bestSlot to compare with yet
                    if (!take) take = bestSlot < 0 || __ldg(&sc.tri_orig[s]) < __ldg(&sc.tri_orig[bestSlot]);
                }
                if (take) {
                    r.bestT = dst; bestU = u; bestV = v; bestSlot = s;
                }
            }
        }
    };
    auto test_leaf = [&](int32_t code) {
        const int32_t packed = ~code;
        const int32_t first = packed & kLeafFirstMask;
        const int32_t cnt = (packed >> kLeafCountShift) + 1;
        for (int32_t s = first; s < first + cnt; s++) {
            if constexpr (ANY) {
                if (bestSlot >= 0) break;  // answered: the rest of the leaf (and a second leaf) is not tested
            }
            test_tri(s);
        }
    };
    // ANY: a ray that accepted a triangle is done.  Its stack and parked leaf are dropped, and the pop phase writes
    // the result and hands the lane to the refill.
    auto any_done = [&]() {
        if constexpr (ANY) {
            if (bestSlot >= 0) { sp = 0; post = kNoLeaf; node = kPop; }
        }
    };
    // (Round 2 measured the two leaves of a lane as ONE merged triangle sequence — the warp iterates max(cntA + cntB)
    // instead of max(cntA) + max(cntB): 5781 vs 5853 Mrays/s, the per-iteration select costs more than the shorter loop
    // saves; profiles/r2_leafmerge_shadeocc_ab.txt.)
    // one stack entry; entries that can no longer hold a hit are dropped
    auto pop_one = [&]() {
        --sp;
        float tn;
        int32_t c;
        st.get(sp, c, tn);
        if (tn <= r.bestT * kWiden) node = c;
    };
    auto postpone = [&]() {
        if (SPEC && is_leaf_code(node) && post == kNoLeaf) {
            post = node;
            node = kPop;
        }
    };
    // one iteration of the node phase for a lane: take the next pending subtree if the lane has none (entries
    // behind the best hit are dropped), then one node step.  Written with selects, not branches.
    auto node_iter_impl = [&](auto deepTag, float bestW) {
        constexpr bool DEEP = decltype(deepTag)::value;
        if (SPEC) {
            const bool doPop = (node == kPop) & (sp > 0);
            sp -= doPop ? 1 : 0;
            int32_t c = kPop;
            float tn = 0.0f;
            if (doPop) st.template getT<DEEP>(sp, c, tn);
            node = (doPop & (tn <= bestW)) ? c : node;
            const bool park = is_leaf_code(node) & (post == kNoLeaf);
            post = park ? node : post;
            node = park ? kPop : node;
        }
        if (node >= 0) {
            if (COUNT) visits++;
            if (WIDE) node_step4<DEEP, WIDEN>(sc, r, node, sp, st);
            else node_step<DEEP, WIDEN>(sc, r, node, sp, st);
            if (SPEC) {
                const bool park = is_leaf_code(node) & (post == kNoLeaf);
                post = park ? node : post;
                node = park ? kPop : node;
            }
        }
    };

    for (;;) {
        // ---- pop phase: lanes that finished a subtree take the next one that can still hold a hit
        if (node == kPop) {
            if (sp == 0) {
                if (SPEC && post != kNoLeaf) {
                    node = kDrain;
                } else {
                    write_result(ray);
                    node = kIdle;
                }
            } else {  // (leaving this pop to the node iterations' select-based one: -1.9 %, the vote below needs it)
                pop_one();
                postpone();
            }
        }
        // ---- refill idle lanes from the queue
        uint32_t idle = __ballot_sync(FULL, node == kIdle);
        if (!exhausted && ((int)__popc(idle) >= kRefill || idle == FULL)) {
            // The warp owns a private range [next, end) of the queue, claimed kExtClaim rays at a time: one atomic on
            // the shared cursor per chunk instead of one per refill, and a refill out of the private range waits for no
            // atomic at all.  The leftover of a range is handed out before the fresh chunk, so no ray is skipped.
            uint32_t* const cl = sClaim[threadIdx.x >> 5];
            const uint32_t next = cl[0], end = cl[1], gdone = cl[2];
            const uint32_t want = __popc(idle);
            const uint32_t avail = end - next;
            const bool fresh = avail < want && gdone == 0u;  // warp-uniform
            uint32_t fbase = 0, fend = 0;
            if (fresh) {
                const int leader = __ffs(idle) - 1;
                if ((int)lane == leader) fbase = atomicAdd(cursor, kExtClaim);
                fbase = __shfl_sync(FULL, fbase, leader);
                fbase = min(fbase, n);
                fend = min(fbase + kExtClaim, n);
            }
            if (node == kIdle) {
                const uint32_t rank = __popc(idle & ltMask);
                uint32_t i = next + rank;
                bool have = rank < avail;
                if (!have && fresh) {
                    i = fbase + (rank - avail);
                    have = i < fend;
                }
                if (have) {
                    ray = i;
                    bool live = true;
                    if constexpr (Q == Query::RENDER) {
                        const float4 a = cur.od0[i];
                        const float4 b = cur.od1[i];
                        r.o = v3(a.x, a.y, a.z);
                        r.d = v3(a.w, b.x, b.y);
                        r.bestT = kMissT;
                    } else {
                        // 12-byte records: 32 consecutive rays of a warp read 384 contiguous bytes per array
                        const size_t k = 3 * (size_t)i;
                        r.o = v3(qa.o3[k], qa.o3[k + 1], qa.o3[k + 2]);
                        r.d = v3(qa.d3[k], qa.d3[k + 1], qa.d3[k + 2]);
                        const float tm = qa.tmax ? qa.tmax[i] : kMissT;
                        // NaN, zero or negative tmax: no hit possible, the ray is not traversed.  (fminf in slab1
                        // would ignore a NaN bound, so it must not reach bestT.)
                        live = tm > 0.0f;
                        const float bound = fminf(tm, kMissT);
                        r.bestT = __int_as_float(__float_as_int(bound) - 1);  // largest float below the bound
                    }
                    r.g = make_grid_ray(sc, r.o, r.d);
                    bestU = 0.0f; bestV = 0.0f; bestSlot = -1;
                    sp = 0;
                    post = kNoLeaf;
                    node = sc.root_is_leaf ? pack_leaf(0, sc.num_tris) : 0;
                    if (!live) node = kPop;
                    postpone();
                }
            }
            uint32_t nnext, nend, ndone = gdone;
            if (fresh) {
                nnext = min(fbase + (want - avail), fend);
                nend = fend;
                if (fend >= n) ndone = 1u;
            } else {
                nnext = next + min(want, avail);
                nend = end;
            }
            if (Q == Query::RENDER && lane < 10u) {
                // the records this warp takes at its NEXT refill are known exactly: the head of its private range
                // (five 128-byte lines of each array cover 32 records wherever the range starts).  The queries do
                // not prefetch.
                const uint32_t p = nnext + 8u * (lane < 5u ? lane : lane - 5u);
                const void* q = lane < 5u ? (const void*)&cur.od0[p] : (const void*)&cur.od1[p];
                if (p < nend) prefetch_l2(q);
            }
            __syncwarp();
            if (lane == 0) { cl[0] = nnext; cl[1] = nend; cl[2] = ndone; }
            __syncwarp();
            if (ndone != 0u && nnext == nend) exhausted = true;
            idle = __ballot_sync(FULL, node == kIdle);
        }
        if (idle == FULL) {
            if (exhausted) break;
            continue;
        }
        // ---- vote: leaf step or node steps (warp-uniform branch)
        const bool parked = is_leaf_code(node) || node == kDrain;
        const uint32_t parkedM = __ballot_sync(FULL, parked);
        const uint32_t nodeM = __ballot_sync(FULL, node >= 0 || (SPEC && node == kPop));
        if ((int)__popc(parkedM) >= kLeafVote || nodeM == 0u) {
            if (SPEC) {
                if (post != kNoLeaf) {
                    test_leaf(post);
                    if (is_leaf_code(node)) test_leaf(node);
                    post = kNoLeaf;
                    if (parked) node = kPop;
                    any_done();
                }
            } else if (parked) {
                test_leaf(node);
                node = kPop;
                any_done();
            }
        } else {
            // several node steps per vote amortise the voting overhead.  When no lane can reach the end of the
            // shared part of its stack within this round, the loop without any overflow code runs.
            const bool deep = __any_sync(FULL, sp + (WIDE ? 3 : 1) * kNodeSteps >= kShStack);
            const float bestW = r.bestT * kWiden;
            if (!deep) {
#pragma unroll 1
                for (int k = 0; k < kNodeSteps; k++) node_iter_impl(std::false_type{}, bestW);
            } else {
#pragma unroll 1
                for (int k = 0; k < kNodeSteps; k++) node_iter_impl(std::true_type{}, bestW);
            }
        }
    }
    if (COUNT) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            visits += __shfl_xor_sync(FULL, visits, off);
            tests += __shfl_xor_sync(FULL, tests, off);
        }
        if (lane == 0) {
            atomicAdd(&stats[2], (unsigned long long)visits);
            atomicAdd(&stats[3], (unsigned long long)tests);
        }
    }
}

// The random numbers one bounce consumes (S:503-552): the rejection-sampled unit vector (3 draws per
// try) when the material scatters diffusely, then `nExtra` more draws (specular choice, Russian roulette).
struct BounceRandoms {
    V3 randDir;
    float d0, d1;
};
constexpr int kCoopOwners = 10;  // RT_RNG_PHILOX: pending lanes served per stage-2 pass (3 blocks each: 30 of the 32 lanes work)
struct CoopSlot {
    uint32_t pixel, frame, sample, pad;
};
// RT_RNG_REF_PCG: the reference's sequential stream, drawn exactly in shader order.
__device__ __forceinline__ BounceRandoms bounce_randoms(Rng<0>& rng, bool needDir, int nExtra, CoopSlot*) {
    BounceRandoms r;
    r.randDir = v3(0.0f, 0.0f, 0.0f);
    r.d0 = r.d1 = 0.0f;
    if (needDir) r.randDir = random_direction(rng);
    if (nExtra >= 1) r.d0 = rng.next();
    if (nExtra >= 2) r.d1 = rng.next();
    return r;
}
// RT_RNG_PHILOX: draw j of a bounce is a pure function of (pixel, frame, sample, bounce, j): word j & 3 of Philox block
// j >> 2.  Generating a block costs ~70 instructions, and a lane needs blocks only as far as its rejection loop gets
// (S:176-183: 3 draws per try, acceptance 52.4 %, then the 1-2 draws after the accepted try): two blocks for 77 % of
// the lanes, more for the rest.  Round 1 let every lane compute five blocks in lock step (ncu: 9.5 -> 17.6 lanes per
// instruction, but 75 % of k_shade's instructions were Philox rounds).  Now:
//   stage 1  every lane computes blocks 0 and 1 of ITS path and evaluates tries 1 and 2 (draws 0..5, extras up to 7);
//   stage 2  the lanes still without a direction (7 of 32 on average) hand their key to the warp through shared
//            memory, and lane L computes block 2 + L % 3 FOR pending lane number L / 3: one block-time of the whole
//            warp produces the three further blocks of up to ten paths; each owner collects its twelve words with
//            shuffles and evaluates tries 3..6 (draws 6..17, extras up to 19);
//   tail     the 1.2 % whose six tries all fail continue sequentially from draw 18 as before.
// Values and draw indices are those of the sequential definition, so no bit of the image changes.
// The acceptance test of S:180, `length(v) < 1`, is evaluated as `dot(v, v) < 1`: sqrt is correctly rounded and
// monotonic, the largest float below 1 is 1 - 2^-24 and sqrt(1 - 2^-24) = 1 - 2^-25 - 2^-51 - ... lies below the
// midpoint of (1 - 2^-24, 1), so it rounds to a value < 1; for x >= 1, sqrt(x) >= 1.  Same decision, no sqrt
// (tests/test_oracle_cpu.py::test_rejection_test_without_sqrt).
__device__ __forceinline__ BounceRandoms bounce_randoms(Rng<1>& rng, bool needDir, int nExtra, CoopSlot* sWarp) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31u;
    BounceRandoms r;
    r.randDir = v3(0.0f, 0.0f, 0.0f);
    // The draws stay 32-bit words until they are used: a candidate component is one I2F + one FFMA
    // (u32_to_signed_unit), and only the two extra draws that are finally selected are converted to [0, 1).
    uint32_t w[8];
    philox4x32_10(0u, rng.bounce, rng.sample, 0x52543230u, rng.pixel, rng.frame, w);
    if (!__any_sync(FULL, needDir)) {  // a warp of glass (or finished) paths: draws 0 and 1 only
        r.d0 = u32_to_unit(w[0]);
        r.d1 = u32_to_unit(w[1]);
        return r;
    }

    // ---- stage 1: blocks 0 and 1, tries 1 and 2
    philox4x32_10(1u, rng.bounce, rng.sample, 0x52543230u, rng.pixel, rng.frame, w + 4);
    bool found = false;
    V3 c = v3(0.0f, 0.0f, 0.0f);
    uint32_t e0 = w[0], e1 = w[1];  // the extra draws of a lane that needs no direction
#pragma unroll
    for (int t = 0; t < 2; t++) {
        const V3 cand = v3(u32_to_signed_unit(w[3 * t]), u32_to_signed_unit(w[3 * t + 1]), u32_to_signed_unit(w[3 * t + 2]));
        const bool acc = needDir && !found && dot(cand, cand) < 1.0f;
        if (acc) {
            c = cand;
            e0 = w[3 * t + 3];
            e1 = w[3 * t + 4];
        }
        found = found || acc;
    }
    // ---- stage 2: the pending lanes' blocks 2, 3, 4 computed by the whole warp, kCoopOwners paths per pass
    bool pending = needDir && !found;
    uint32_t last[4] = {0u, 0u, 0u, 0u};  // block 4 of a lane that goes on to the sequential tail
    bool exhausted = false;               // all six tries failed
    for (uint32_t U = __ballot_sync(FULL, pending); U != 0u; U = __ballot_sync(FULL, pending)) {
        const uint32_t rank = (uint32_t)__popc(U & ((1u << lane) - 1u));
        const bool owner = pending && rank < (uint32_t)kCoopOwners;
        const uint32_t served = min((uint32_t)__popc(U), (uint32_t)kCoopOwners);
        if (owner) sWarp[rank] = CoopSlot{rng.pixel, rng.frame, rng.sample, 0u};
        __syncwarp();
        uint32_t wj[4] = {0u, 0u, 0u, 0u};
        const uint32_t job = lane / 3u;
        if (job < served) {
            const CoopSlot key = sWarp[job];
            philox4x32_10(2u + (lane - 3u * job), rng.bounce, key.sample, 0x52543230u, key.pixel, key.frame, wj);
        }
        __syncwarp();  // the slots are rewritten by the next pass
        // draws 6..19 of an owner: 6, 7 from its own block 1, 8..19 from lanes 3 rank .. 3 rank + 2
        uint32_t g[14];
        g[0] = w[6];
        g[1] = w[7];
        const uint32_t src = owner ? 3u * rank : lane;
#pragma unroll
        for (int b = 0; b < 3; b++) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t v = __shfl_sync(FULL, wj[k], (src + b) & 31u);
                g[2 + 4 * b + k] = v;
                if (b == 2) last[k] = owner ? v : last[k];
            }
        }
        if (owner) {
#pragma unroll
            for (int t = 0; t < 4; t++) {  // tries 3..6: draws 6 + 3 t .. 8 + 3 t, extras 9 + 3 t and 10 + 3 t
                const V3 cand = v3(u32_to_signed_unit(g[3 * t]), u32_to_signed_unit(g[3 * t + 1]), u32_to_signed_unit(g[3 * t + 2]));
                const bool acc = !found && dot(cand, cand) < 1.0f;
                if (acc) {
                    c = cand;
                    e0 = g[3 * t + 3];
                    e1 = g[3 * t + 4];
                }
                found = found || acc;
            }
            exhausted = !found;
            pending = false;
        }
    }
    r.d0 = u32_to_unit(e0);
    r.d1 = u32_to_unit(e1);
    if (needDir) {
        if (found) {
            r.randDir = normalize(c);
        } else if (exhausted) {
            // tries 7..100 of S:176-183, sequentially, from draw 18 (block 4 is already in hand)
            rng.j = 18u;
            rng.cache[0] = last[0]; rng.cache[1] = last[1]; rng.cache[2] = last[2]; rng.cache[3] = last[3];
            for (int i = 6; i < 100; i++) {
                const float x = rng.next() * 2.0f - 1.0f;
                const float y = rng.next() * 2.0f - 1.0f;
                const float z = rng.next() * 2.0f - 1.0f;
                if (dot(v3(x, y, z), v3(x, y, z)) < 1.0f) {
                    r.randDir = normalize(v3(x, y, z));
                    break;
                }
            }
            if (nExtra >= 1) r.d0 = rng.next();
            if (nExtra >= 2) r.d1 = rng.next();
        }
    }
    return r;
}

// ---------------------------------------------------------------------------------------------- k_shade
// Not split per material.  Round 2 built block-local material queues (every block sorted the 256 paths of its window
// by material class with warp ballots + a prefix over the (warp, class) counts, and appended its survivors ordered by
// the octant of their new direction with one atomicAdd per block) and measured them on config 2, B200, same run:
// plain kernel 4995 Mrays/s; class queues 4762 (-4.7 %); octant-ordered block output 4803 (-3.8 %, k_extend unchanged
// at 7.93 ms per launch: ray octants at block granularity buy no coherence); both 4632 (-7.3 %) — raw lines in
// profiles/r2_shade_queues_ab.txt, code in commit c59b9e8.  The sort's barriers and its uncoalesced (sorted) loads cost
// more than the divergence they remove: DIFFUSE and TEXTURE share the switch case, so on this workload only the
// texture fetch diverges.  What is kept from that work: the random numbers of a bounce are drawn by the converged
// warp, and a warp whose paths all end (miss, light, unknown material) draws none.
// One bounce of S:481-560 for every live path.  `bounce` is the 0-based index of this segment.
// Measured and not kept (profiles/r2_final_ab.txt): survivors appended with one atomicAdd per BLOCK window (warp counts
// scanned in shared memory between two barriers) instead of one per warp: config 2 5604 vs 5854 Mrays/s (-4.3 %),
// config 4 4219 vs 4280 — eight times fewer atomics, but every warp of the block then waits at two barriers for the
// block's slowest warp AND for the atomic.  What ships is the deferred append below, which takes the wait off the
// critical path first and then cuts the number of atomics by three without any barrier.
// Measured neutral and removed (profiles/r2_final_ab.txt, code in commit 38eb466): a 256-entry shared-memory table for
// the texel byte -> float conversion (6023 vs 6056 Mrays/s) and warp-cooperative bilinear taps — the textured lanes
// (5 of 32 at the later bounces, a fifth of k_shade's instructions) only prepare the sample and lane L fetches tap
// L % 4 of sample L / 4 — 6056-6067 vs 6048-6058: those bounces wait on their dependent gathers, not on issue slots.
// Also measured and removed (profiles/r2_final_ab.txt): gathering the NEXT window's hit-triangle record into L1 / L2
// while this one is shaded (config 2 6039 / 6029 vs 6049-6059, config 4 +0.9 %), three resident blocks at 80 registers
// without spills (6018), a smaller shade grid (32 / 16 blocks per SM: 6030 / 5981).
constexpr int kShadeMinBlocks = 4;  // 64 registers; 5 blocks (48 registers, 358 B of spills) -15 %, 6 blocks -16 % (profiles/r2_leafmerge_shadeocc_ab.txt)
// Windows per deferred queue reservation.  Measured on four boxes (profiles/r2_final_ab.txt): config 2, bounce 0
// deferred, 1 / 2 / 3 / 4 windows 6059-6066 / 6077 / 6115-6128 / 6063 Mrays/s on every box; config 4, every bounce
// deferred, 1 window 4146 / 4410 / 4540 / 4542 depending on the box (the atomic's latency and rate are the box lottery
// of DESIGN.md section 6.1), 2 windows 4229 / 4257 / 4515, 3 windows 4449 / 4454 / 4461 on all of them, 4 windows
// (48 KB of staging per block: too little L1 left) 4179.
constexpr int kDeferWindows = 3;
template <int MODE, bool DEFER>
__global__ void __launch_bounds__(kBlock, kShadeMinBlocks) k_shade(const __grid_constant__ SceneView sc,
                                                  const __grid_constant__ FrameParams fp, PathArrays cur,
                                                  PathArrays next, const float4* __restrict__ hit,
                                                  float4* __restrict__ contrib, uint32_t* __restrict__ pix_rng,
                                                  const uint32_t* __restrict__ countIn,
                                                  uint32_t* __restrict__ countOut, int bounce) {
    __shared__ CoopSlot sCoop[kBlock / 32][kCoopOwners];  // stage 2 of bounce_randoms: keys handed to the warp
    // DEFER: the survivors of kDeferWindows consecutive windows wait in shared memory, every lane in its own slot,
    // while the warp's ONE queue reservation for them is in flight
    constexpr int kWin = DEFER ? kDeferWindows : 1;
    extern __shared__ float4 sStageDyn[];  // [kDeferWindows][3][kBlock], sized at launch (12 KB per window)
#define sStage(k, c) sStageDyn[((k) * 3 + (c)) * kBlock + threadIdx.x]
    const uint32_t n = *countIn;
    const uint32_t lane = threadIdx.x & 31u;
    constexpr uint32_t FULL = 0xffffffffu;
    uint32_t pend[kWin];  // survivor masks of the windows of the batch being staged / in flight
#pragma unroll
    for (int k = 0; k < kWin; k++) pend[k] = 0u;
    uint32_t pendRaw = 0u, phase = 0u;  // lane 0: the atomicAdd result; which window of the batch comes next
    // the batch in flight goes to the queue: window k of it behind the survivors of windows 0 .. k-1
    auto flush = [&]() {
        uint32_t any = 0u;
#pragma unroll
        for (int k = 0; k < kWin; k++) any |= pend[k];
        if (any == 0u) return;
        uint32_t at = __shfl_sync(FULL, pendRaw, 0);
#pragma unroll
        for (int k = 0; k < kWin; k++) {
            if ((pend[k] >> lane) & 1u) {
                const uint32_t pos = at + __popc(pend[k] & ((1u << lane) - 1u));
                next.od0[pos] = sStage(k, 0);
                next.od1[pos] = sStage(k, 1);
                next.misc[pos] = sStage(k, 2);
            }
            at += __popc(pend[k]);
        }
    };
    auto reserve = [&]() {
        uint32_t total = 0u;
#pragma unroll
        for (int k = 0; k < kWin; k++) total += __popc(pend[k]);
        if (total != 0u && lane == 0u) pendRaw = atomicAdd(countOut, total);
    };
    for (uint32_t base = blockIdx.x * kBlock; base < n; base += gridDim.x * kBlock) {
        const uint32_t i = base + threadIdx.x;
        const bool valid = i < n;
        bool alive = false;
        V3 o = v3(0, 0, 0), d = v3(0, 0, 1), rayColor = v3(0, 0, 0);
        int32_t slotId = 0, hslot = -1, pixLocal = 0, batchFrame = 0;
        uint32_t carry = 0, flags = 0;
        bool insideGlass = false;
        float4 h = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        float4 g3 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // unit normal + material index of the hit triangle
        Material m;
        m.type = -1;
        Rng<MODE> rng;
        rng.init(0u, 0u, 0u, 0u);
        const int bounceCount = bounce + 1;  // S:483
        if (valid) {
            const float4 a = cur.od0[i], b = cur.od1[i], c = cur.misc[i];
            h = hit[i];
            o = v3(a.x, a.y, a.z);
            d = v3(a.w, b.x, b.y);
            rayColor = v3(b.z, b.w, c.x);
            slotId = __float_as_int(c.y);
            carry = __float_as_uint(c.z);
            flags = __float_as_uint(c.w);
            insideGlass = (flags >> 16) & 1u;
            const int slotLane = (int)fastdiv((uint32_t)slotId, fp.div_pixels);
            pixLocal = slotId - slotLane * fp.local_pixels;
            batchFrame = fp.frames_in_batch > 1 ? (int)fastdiv((uint32_t)slotLane, fp.div_samples) : 0;
            rng.init(carry, local_pixel_id(fp, pixLocal), fp.u.frameIndex + (uint32_t)(batchFrame * fp.frame_stride), 0u);
            hslot = __float_as_int(h.w);
            if (hslot >= 0) {
                g3 = __ldg(&sc.tri_geom[4 * hslot + 3]);
                m = load_material(sc, __float_as_int(g3.w));
            }
        }
        rng.stream((uint32_t)bounceCount);
        const bool needDir = hslot >= 0 && (m.type == RT_MAT_DIFFUSE || m.type == RT_MAT_TEXTURE ||
                                            m.type == RT_MAT_SPECULAR || m.type == RT_MAT_CHECKER);
        const int nExtra = (hslot < 0) ? 0 : (m.type == RT_MAT_SPECULAR ? 2 : ((needDir || m.type == RT_MAT_GLASS) ? 1 : 0));
        // the random numbers of the bounce, drawn by the whole warp together (lock-step Philox blocks); a warp of
        // terminal paths draws nothing
        BounceRandoms rnd;
        rnd.randDir = v3(0.0f, 0.0f, 0.0f);
        rnd.d0 = rnd.d1 = 0.0f;
        if (MODE == 0 || __any_sync(FULL, needDir || nExtra > 0))
            rnd = bounce_randoms(rng, needDir, nExtra, sCoop[threadIdx.x >> 5]);
        if (valid) {
            bool terminated = false;
            V3 radiance = v3(0.0f, 0.0f, 0.0f);
            if (hslot >= 0) {
                const float dst = h.x, bu = h.y, bv = h.z;
                const V3 hitPoint = o + d * dst;        // S:330
                const V3 normal = v3(g3.x, g3.y, g3.z);  // S:331
                if (m.type != RT_MAT_GLASS)
                    o = hitPoint - (d * dst) * -1e-3f;  // S:490
                else
                    o = hitPoint + (d * dst) * -1e-3f;  // S:492
                V3 attenuation = v3(0.0f, 0.0f, 0.0f);
                const V3 prevDirection = d;
                float rrDraw = rnd.d0;
                switch (m.type) {
                    case RT_MAT_DIFFUSE:
                    case RT_MAT_TEXTURE: {
                        d = normalize(normal + rnd.randDir);
                        if (m.type == RT_MAT_DIFFUSE)
                            attenuation = m.color;
                        else
                            attenuation = triangle_texture_color(sc, fp.u.numTextures, m.textureIndex,
                                                                 (1.0f - bu) - bv, bu, bv, hslot);
                        break;
                    }
                    case RT_MAT_SPECULAR: {
                        const V3 diffuseDirection = normalize(normal + rnd.randDir);
                        const V3 specularDirection = reflect(d, normal);
                        const bool isSpecularBounce = m.specularProbability > rnd.d0;
                        d = mix(diffuseDirection, specularDirection, isSpecularBounce ? m.smoothness : 0.0f);
                        attenuation = isSpecularBounce ? v3(1.0f, 1.0f, 1.0f) : m.color;
                        rrDraw = rnd.d1;
                        break;
                    }
                    case RT_MAT_LIGHT: {
                        const V3 emitted = m.emission * m.emissionStrength;
                        radiance = v3(0.0f, 0.0f, 0.0f) + emitted * rayColor;  // S:516-517
                        terminated = true;
                        break;
                    }
                    case RT_MAT_CHECKER: {
                        d = normalize(normal + rnd.randDir);
                        attenuation = black_checker(o, m.checkerScale) ? v3(0.0f, 0.0f, 0.0f) : v3(1.0f, 1.0f, 1.0f);
                        break;
                    }
                    case RT_MAT_GLASS: {
                        const float ri = insideGlass ? m.refractiveIndex : 1.0f / m.refractiveIndex;
                        bool isRefracted;
                        d = refract_(d, normal, ri, isRefracted);
                        insideGlass = isRefracted != insideGlass;
                        attenuation = m.color;
                        break;
                    }
                    default:
                        radiance = v3(1.0f, 0.0f, 1.0f);  // S:540
                        terminated = true;
                        break;
                }
                if (!terminated) {
                    if (m.isEdgeHighlight != 0 && bounceCount > 1)
                        d = prevDirection;
                    else
                        rayColor = rayColor * attenuation;
                    const float p = gmax(rayColor.x, gmax(rayColor.y, rayColor.z));  // S:549-552
                    if (rrDraw > p) {
                        terminated = true;
                    } else {
                        rayColor = rayColor * (1.0f / p);
                        if (bounceCount >= fp.u.maxBounceCount) terminated = true;  // loop condition S:481
                    }
                }
            } else {
                if (fp.u.environmentalLight != 0) radiance = v3(0.0f, 0.0f, 0.0f) + env_light(d) * rayColor;
                terminated = true;
            }
            carry = rng.carry();
            if (terminated) {
                contrib[slotId] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
                // the pixel's stream continues with the next sample of the same frame
                if (MODE == 0) pix_rng[(size_t)batchFrame * fp.local_pixels + pixLocal] = carry;
            } else {
                alive = true;
                flags = (uint32_t)bounceCount | ((insideGlass ? 1u : 0u) << 16);
            }
        }
        // compaction: the survivors of this warp take consecutive places in the next queue
        const uint32_t mask = __ballot_sync(FULL, alive);
        if (DEFER) {
            // Deferred append.  The warp's atomicAdd on the queue counter takes microseconds to return, and the 4.2 M of
            // them per 133 M-path launch all hit one address (ncu, v19: 41.6 % of k_shade's stall samples at bounce 0
            // of config 2 and 44 % at every bounce of config 4 sat on the shuffle that broadcasts the result).  So the
            // survivors of kDeferWindows consecutive windows share ONE reservation, issued when the last of them is staged,
            // and are written to the queue at the end of the window after that — a whole iteration later.
            if (phase == 0u) {
                flush();
#pragma unroll
                for (int k = 0; k < kWin; k++) pend[k] = 0u;
            }
#pragma unroll
            for (int k = 0; k < kWin; k++)
                if ((uint32_t)k == phase) pend[k] = mask;
            if (alive) {
                sStage(phase, 0) = make_float4(o.x, o.y, o.z, d.x);
                sStage(phase, 1) = make_float4(d.y, d.z, rayColor.x, rayColor.y);
                sStage(phase, 2) = make_float4(rayColor.z, __int_as_float(slotId), __uint_as_float(carry),
                                               __uint_as_float(flags));
            }
            phase = phase + 1u == (uint32_t)kWin ? 0u : phase + 1u;
            if (phase == 0u) reserve();
        } else {
            uint32_t basePos = 0;
            if (mask) {
                const int leader = __ffs(mask) - 1;
                if ((int)lane == leader) basePos = atomicAdd(countOut, (uint32_t)__popc(mask));
                basePos = __shfl_sync(FULL, basePos, leader);
            }
            const uint32_t pos = basePos + __popc(mask & ((1u << lane) - 1u));
            if (alive) {
                next.od0[pos] = make_float4(o.x, o.y, o.z, d.x);
                next.od1[pos] = make_float4(d.y, d.z, rayColor.x, rayColor.y);
                next.misc[pos] = make_float4(rayColor.z, __int_as_float(slotId), __uint_as_float(carry),
                                             __uint_as_float(flags));
            }
        }
    }
    if (DEFER) {
        if (phase != 0u) reserve();  // an incomplete last batch has no reservation yet
        flush();
    }
}
#undef sStage

__global__ void __launch_bounds__(kBlock) k_accumulate(const __grid_constant__ FrameParams fp,
                                                       const float4* __restrict__ contrib,
                                                       float4* __restrict__ accum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // (batch frame, local pixel)
    if (i >= fp.local_pixels * fp.frames_in_batch) return;
    const int k = i / fp.local_pixels;
    const int p = i - k * fp.local_pixels;
    float4 acc = accum[i];
    const float4* c0 = contrib + (size_t)k * fp.samples_in_batch * fp.local_pixels + p;
    for (int s = 0; s < fp.samples_in_batch; s++) {  // sample order (S:683-694)
        const float4 c = c0[(size_t)s * fp.local_pixels];
        acc.x = acc.x + c.x;
        acc.y = acc.y + c.y;
        acc.z = acc.z + c.z;
    }
    accum[i] = acc;
}

// One thread per local pixel walks the batch frames in order: the image keeps the last frame (what the
// reference's image binding holds after the last dispatch), the 8-bit sums take every frame (R:217-229).
__global__ void __launch_bounds__(kBlock) k_resolve(const __grid_constant__ FrameParams fp,
                                                    const float4* __restrict__ accum, float4* __restrict__ image,
                                                    uint32_t* __restrict__ frame_sum, int add_to_sum) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= fp.local_pixels) return;
    int tx, ty;
    local_pixel_xy(fp, p, tx, ty);
    const float nr = (float)fp.u.numRaysPerPixel;
    const size_t pix = (size_t)ty * fp.width + tx;
    uint32_t sr = 0, sg = 0, sb = 0;
    V3 color = v3(0.0f, 0.0f, 0.0f);
    for (int k = 0; k < fp.frames_in_batch; k++) {
        const float4 a = accum[(size_t)k * fp.local_pixels + p];
        color = v3(a.x / nr, a.y / nr, a.z / nr);  // S:696
        color = tonemap_srgb(color);               // S:697
        sr += quantize8(color.x);
        sg += quantize8(color.y);
        sb += quantize8(color.z);
    }
    image[pix] = make_float4(color.x, color.y, color.z, 1.0f);  // S:700
    if (add_to_sum) {
        frame_sum[pix * 3 + 0] += sr;
        frame_sum[pix * 3 + 1] += sg;
        frame_sum[pix * 3 + 2] += sb;
    }
}

// R:248-259
__global__ void __launch_bounds__(kBlock) k_finalize(const uint32_t* __restrict__ frame_sum, uint8_t* __restrict__ out,
                                                     int w, int h, int frames) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t rowLen = (size_t)w * 3;
    if (j >= rowLen * h) return;
    const size_t y = j / rowLen, x = j - y * rowLen;
    const float avg = (float)frame_sum[j] / (float)frames;
    const float c = avg < 255.0f ? avg : 255.0f;
    out[(size_t)(h - 1 - y) * rowLen + x] = (uint8_t)c;
}

__device__ __forceinline__ V3 normalize_color(V3 c) {  // S:462-470
    const float m = gmax(gmax(c.x, c.y), c.z);
    if (m > 1.0f) return c / m;
    return c;
}

// S:565-645: preview shading, deterministic centre ray, one thread per pixel
__global__ void __launch_bounds__(kBlock) k_preview(const __grid_constant__ SceneView sc,
                                                    const __grid_constant__ FrameParams fp,
                                                    float4* __restrict__ image,
                                                    unsigned long long* __restrict__ stats) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= fp.local_pixels) return;
    int tx, ty;
    local_pixel_xy(fp, p, tx, ty);
    const PixelSetup ps = pixel_setup(fp.u, tx, ty);
    V3 o = v3(fp.u.cameraPos), d = ps.centreDir;
    bool insideGlass = false;
    V3 cum = v3(0.0f, 0.0f, 0.0f);
    int bounceCount = 0;
    uint32_t segs = 0;
    V3 result = v3(0.0f, 0.0f, 0.0f);
    bool done = false;
    while (bounceCount < fp.u.maxBounceCount && !done) {
        bounceCount++;
        const HitRec h = closest_hit(sc, o, d);
        segs++;
        if (h.slot >= 0) {
            const V3 hitPoint = o + d * h.t;
            const V3 normal = tri_normal(sc, h.slot);
            o = hitPoint - normal * 1e-4f;
            const float4 s1 = __ldg(&sc.tri_shade[2 * h.slot + 1]);
            const Material m = load_material(sc, __float_as_int(s1.z));
            switch (m.type) {
                case RT_MAT_SPECULAR:
                    cum = cum + m.color;
                    d = reflect(d, normal);
                    break;
                case RT_MAT_DIFFUSE:
                case RT_MAT_TEXTURE:
                case RT_MAT_CHECKER: {
                    V3 color;
                    if (m.type == RT_MAT_TEXTURE)
                        color = triangle_texture_color(sc, fp.u.numTextures, m.textureIndex, (1.0f - h.u) - h.v,
                                                       h.u, h.v, h.slot);
                    else if (m.type == RT_MAT_DIFFUSE)
                        color = m.color;
                    else
                        color = black_checker(o, m.checkerScale) ? v3(0.0f, 0.0f, 0.0f) : v3(1.0f, 1.0f, 1.0f);
                    cum = cum + color;
                    if (fp.u.basicShadingShadow != 0) {
                        const V3 toLight = normalize(v3(fp.u.basicShadingLightPosition) - hitPoint);
                        const HitRec sh = closest_hit(sc, o, toLight);
                        segs++;
                        const V3 c = sh.slot >= 0 ? cum / 5.0f : cum;
                        result = c / (float)bounceCount;
                    } else {
                        result = cum / (float)bounceCount;
                    }
                    done = true;
                    break;
                }
                case RT_MAT_LIGHT:
                    result = normalize_color(m.emission);
                    done = true;
                    break;
                case RT_MAT_GLASS: {
                    const float ri = insideGlass ? m.refractiveIndex : 1.0f / m.refractiveIndex;
                    bool isRefracted;
                    d = refract_(d, normal, ri, isRefracted);
                    insideGlass = isRefracted != insideGlass;
                    cum = m.color;
                    break;
                }
                case RT_MAT_GLASS_HIGHLIGHT:
                    break;
                default:
                    result = v3(1.0f, 0.0f, 1.0f);
                    done = true;
                    break;
            }
        } else {
            cum = cum + env_light(d);
            break;
        }
    }
    if (!done) result = cum / (float)bounceCount;
    image[(size_t)ty * fp.width + tx] = make_float4(result.x, result.y, result.z, 1.0f);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) segs += __shfl_xor_sync(0xffffffffu, segs, off);
    if ((threadIdx.x & 31) == 0) atomicAdd(&stats[0], (unsigned long long)segs);
}

// ---- parity hooks.  rt_first_hit and rt_trace_rays are the closest-hit query (wf_query, Query::CLOSEST) on staged
// copies; this kernel writes rt_first_hit's camera rays as the (N, 3) origin and direction arrays the query reads.
template <int MODE>
__global__ void __launch_bounds__(kBlock) k_first_rays(const __grid_constant__ FrameParams fp, int mode,
                                                       float* __restrict__ o3, float* __restrict__ d3) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= fp.width * fp.height) return;
    const int ty = p / fp.width, tx = p - ty * fp.width;
    const PixelSetup ps = pixel_setup(fp.u, tx, ty);
    V3 o, d;
    if (mode == RT_FIRST_HIT_CENTRE) {
        o = v3(fp.u.cameraPos);
        d = ps.centreDir;
    } else {
        Rng<MODE> rng;
        rng.init(MODE == 0 ? ps.seed : 0u, ps.pixelId, fp.u.frameIndex, 0u);
        rng.stream(0u);
        sample_ray(fp.u, ps, rng, o, d);
    }
    const size_t k = 3 * (size_t)p;  // 64-bit: 3 * p wraps in 32 bits above 715 827 882 pixels
    o3[k] = o.x;
    o3[k + 1] = o.y;
    o3[k + 2] = o.z;
    d3[k] = d.x;
    d3[k + 1] = d.y;
    d3[k + 2] = d.z;
}
// ---- ray queries (wf_query): the ctx's count and cursor words, reset on the stream before each query
__global__ void k_query_reset(uint32_t* counts, uint32_t n) {
    if (threadIdx.x == 0) {
        counts[0] = n;   // rays in the queue
        counts[1] = 0u;  // k_extend's work cursor
    }
}

// tile-split plumbing: compact (own rows only) <-> full-frame layouts of the 8-bit frame sums
__global__ void __launch_bounds__(kBlock) k_rows_copy(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                      const int32_t* __restrict__ rows, int nrows, int rowLen,
                                                      int scatter) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (size_t)nrows * rowLen) return;
    const size_t r = j / rowLen, x = j - r * rowLen;
    const size_t full = (size_t)rows[r] * rowLen + x;
    if (scatter) dst[full] = src[j]; else dst[j] = src[full];
}

// ------------------------------------------------------------------------------------------------ launchers
static inline int nblocks(long long n, int per = kBlock) { return (int)((n + per - 1) / per); }

struct Timed {
    const Launcher& L;
    int tag;
    int slot;
    Timed(const Launcher& l, int t) : L(l), tag(t), slot(-1) {
        if (L.timing && *L.ev_used + 2 <= L.ev_cap) {
            slot = *L.ev_used;
            *L.ev_used += 2;
            L.ev_tag[slot] = tag;
            cudaEventRecord(L.ev_pool[slot], L.st);
        }
    }
    ~Timed() {
        if (slot >= 0) cudaEventRecord(L.ev_pool[slot + 1], L.st);
    }
};

using ExtendKernel = void (*)(SceneView, PathArrays, float4*, const uint32_t*, uint32_t*, unsigned long long*, QueryArgs);
template <bool COUNT, bool WIDE>
static ExtendKernel widened_extend(Query q) {
    if (q == Query::CLOSEST) return k_extend<COUNT, WIDE, true, Query::CLOSEST>;
    if (q == Query::ANY) return k_extend<COUNT, WIDE, true, Query::ANY>;
    return k_extend<COUNT, WIDE, true, Query::RENDER>;
}
// The k_extend instantiation for one launch.  `wide`: the scene has the 4-wide tree.  `widen`: origins may lie far
// outside the quantisation grid (rt_scene.cuh, slab1).
static ExtendKernel extend_kernel(bool instrument, bool wide, bool widen, Query q) {
    // the counted walk and the queries always take the widened slab test: only uninstrumented rendering has a variant
    // without it
    widen |= instrument || q != Query::RENDER;
    if (!widen) return wide ? k_extend<false, true, false, Query::RENDER> : k_extend<false, false, false, Query::RENDER>;
    if (instrument) return wide ? widened_extend<true, true>(q) : widened_extend<true, false>(q);
    return wide ? widened_extend<false, true>(q) : widened_extend<false, false>(q);
}

cudaError_t wf_extend_residency(bool instrument, ExtendResidency* r) {
    for (int q = 0; q < 3; q++)
        for (int w = 0; w < 2; w++)
            for (int wd = 0; wd < 2; wd++) {
                const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                    &r->blocks_per_sm[q][w][wd], extend_kernel(instrument, w, wd, (Query)q), kExtBlock, 0);
                if (e != cudaSuccess) return e;
            }
    return cudaSuccess;
}

// One persistent pass of k_extend over the `*count` rays: the instantiation extend_kernel picks, on a grid sized from
// that instantiation's residency.  RENDER reads `rays` (od0 / od1) and writes `hit`; the queries read and write `qa`.
static void launch_extend(const Launcher& L, const SceneView& sc, bool widen, Query q, const PathArrays& rays,
                          float4* hit, const uint32_t* count, uint32_t* cursor, unsigned long long* stats,
                          const QueryArgs& qa) {
    const bool wide = sc.nodes4 != nullptr;
    const int grid = L.sm_count * L.extend_residency->blocks_per_sm[(int)q][wide][widen];
    extend_kernel(L.instrument, wide, widen, q)<<<grid, kExtBlock, 0, L.st>>>(sc, rays, hit, count, cursor, stats, qa);
    (*L.kernel_launches)++;
    (*L.extend_launches)++;
}

cudaError_t wf_clear_accum(const Launcher& L, const WaveBuffers& wb, long long entries) {
    k_clear_accum<<<nblocks(entries), kBlock, 0, L.st>>>(wb.accum, (int)entries);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

cudaError_t wf_seed_pixels(const Launcher& L, const SceneView&, const WaveBuffers& wb, const FrameParams& fp) {
    k_seed_pixels<<<nblocks((long long)fp.local_pixels * fp.frames_in_batch), kBlock, 0, L.st>>>(fp, wb.pix_rng);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

cudaError_t wf_render_batch(const Launcher& L, const SceneView& sc, const WaveBuffers& wb, const FrameParams& fp) {
    const long long n = (long long)fp.local_pixels * fp.lanes_active;
    const int maxB = fp.u.maxBounceCount;
    const int ncounts = maxB + 2;
    {
        Timed t(L, 1);
        if (L.rng_mode == RT_RNG_REF_PCG)
            k_raygen<0><<<nblocks(n), kBlock, 0, L.st>>>(fp, wb.cur, wb.contrib, wb.pix_rng, wb.counts, ncounts, wb.stats);
        else
            k_raygen<1><<<nblocks(n), kBlock, 0, L.st>>>(fp, wb.cur, wb.contrib, wb.pix_rng, wb.counts, ncounts, wb.stats);
        (*L.kernel_launches)++;
    }
    // fixed-size grids that read the live count on the device: no host round trip per bounce
    const long long gridCap = (long long)L.sm_count * L.shade_blocks_per_sm;
    const int grid = (int)((n + kBlock - 1) / kBlock < gridCap ? (n + kBlock - 1) / kBlock : gridCap);
    uint32_t* cursors = wb.counts + ncounts;
    PathArrays a = wb.cur, b = wb.next;
    for (int bounce = 0; bounce < maxB; bounce++) {
        {
            Timed t(L, 0);
            // camera rays may start far outside the scene; every later segment starts on a surface of it
            launch_extend(L, sc, bounce == 0 && L.widen_primary, Query::RENDER, a, wb.hit, wb.counts + bounce,
                          cursors + bounce, wb.stats, QueryArgs{});
        }
        {
            Timed t(L, 1);
            // Deferred append (see k_shade) at bounce 0 and, when the scene has no textures, at every bounce.  Measured
            // on B200 (profiles/r2_final_ab.txt): bounce 0 is latency-bound everywhere (config 2: +1.5 % from deferring
            // it alone); the later bounces of the textured config-2 scene are issue-bound (66 % issue-active, 17.8 lanes
            // per instruction) and LOSE 0.8-2.4 % to the staging, those of the untextured 10 M-triangle scene wait on
            // the atomic like bounce 0 does (34 % issue-active, 44 % of the stall samples) and gain 3.3-9.4 % depending
            // on the box.
            const bool defer = bounce == 0 || fp.u.numTextures <= 0;
            const size_t stage_bytes = defer ? (size_t)kDeferWindows * 3 * kBlock * sizeof(float4) : 0;
#define RT_SHADE(M, D) k_shade<M, D><<<grid, kBlock, stage_bytes, L.st>>>(sc, fp, a, b, wb.hit, wb.contrib, wb.pix_rng, wb.counts + bounce, \
                                                                        wb.counts + bounce + 1, bounce)
            if (L.rng_mode == RT_RNG_REF_PCG) {
                if (defer) RT_SHADE(0, true); else RT_SHADE(0, false);
            } else {
                if (defer) RT_SHADE(1, true); else RT_SHADE(1, false);
            }
#undef RT_SHADE
            (*L.kernel_launches)++;
        }
        PathArrays tmp = a;
        a = b;
        b = tmp;
    }
    {
        Timed t(L, 1);
        k_accumulate<<<nblocks((long long)fp.local_pixels * fp.frames_in_batch), kBlock, 0, L.st>>>(fp, wb.contrib, wb.accum);
        (*L.kernel_launches)++;
    }
    return cudaGetLastError();
}

cudaError_t wf_resolve_frame(const Launcher& L, const WaveBuffers& wb, const FrameParams& fp, bool add_to_sum) {
    Timed t(L, 1);
    k_resolve<<<nblocks(fp.local_pixels), kBlock, 0, L.st>>>(fp, wb.accum, wb.image, wb.frame_sum, add_to_sum ? 1 : 0);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

cudaError_t wf_preview(const Launcher& L, const SceneView& sc, const WaveBuffers& wb, const FrameParams& fp) {
    Timed t(L, 0);
    k_preview<<<nblocks(fp.local_pixels), kBlock, 0, L.st>>>(sc, fp, wb.image, wb.stats);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

cudaError_t wf_finalize(const Launcher& L, const uint32_t* frame_sum, uint8_t* out, int w, int h, int frames) {
    Timed t(L, 1);
    k_finalize<<<nblocks((long long)w * h * 3), kBlock, 0, L.st>>>(frame_sum, out, w, h, frames);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

cudaError_t wf_first_rays(const Launcher& L, const FrameParams& fp, int mode, float* o3, float* d3) {
    const long long n = (long long)fp.width * fp.height;
    if (L.rng_mode == RT_RNG_REF_PCG)
        k_first_rays<0><<<nblocks(n), kBlock, 0, L.st>>>(fp, mode, o3, d3);
    else
        k_first_rays<1><<<nblocks(n), kBlock, 0, L.st>>>(fp, mode, o3, d3);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

// The ray queries run k_extend straight on the arrays they are given: one tiny kernel resets the ctx's count and cursor
// words on the stream, then the persistent traversal.  No staging, no copy, no host synchronisation.
cudaError_t wf_query(const Launcher& L, const SceneView& sc, const QueryArgs& q, int64_t n, Query mode,
                     uint32_t* counts, unsigned long long* stats) {
    if (n <= 0) return cudaSuccess;
    k_query_reset<<<1, 32, 0, L.st>>>(counts, (uint32_t)n);
    (*L.kernel_launches)++;
    launch_extend(L, sc, true, mode, PathArrays{nullptr, nullptr, nullptr}, nullptr, counts, counts + 1, stats, q);
    return cudaGetLastError();
}

cudaError_t wf_scatter_rows(const Launcher& L, const uint32_t* compact, uint32_t* full, const int32_t* rows, int nrows,
                            int width) {
    if (nrows <= 0) return cudaSuccess;
    k_rows_copy<<<nblocks((long long)nrows * width * 3), kBlock, 0, L.st>>>(compact, full, rows, nrows, width * 3, 1);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}
cudaError_t wf_gather_rows(const Launcher& L, const uint32_t* full, uint32_t* compact, const int32_t* rows, int nrows,
                           int width) {
    if (nrows <= 0) return cudaSuccess;
    k_rows_copy<<<nblocks((long long)nrows * width * 3), kBlock, 0, L.st>>>(full, compact, rows, nrows, width * 3, 0);
    (*L.kernel_launches)++;
    return cudaGetLastError();
}

}  // namespace rt
