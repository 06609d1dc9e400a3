/*
 * rt_b200.h — C-ABI of the B200-native path-tracing backend (librt_b200.so).
 *
 * This header is the drop-in boundary for the ONE hot path of
 * jackbaggins/RayTracing2-fork: the per-pixel path tracer that the reference runs as the
 * OpenGL compute shader RayTracing/Assets/Shaders/compute.glsl, plus the CPU BVH build in
 * front of it and the screenshot accumulation behind it.  The reference has no FFI; its de-facto
 * operator interface is the GL binding table (3 SSBOs, 1 UBO, <=5 samplers, 1 image) and the two
 * dispatch sites.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference tree).
 *
 * Rules of the boundary
 *   - plain C, plain pointers and sizes; no exceptions, no C++ or torch types cross it;
 *   - every call returns an int status (RT_OK == 0); rt_last_error(ctx) gives the text;
 *   - CUDA / NCCL errors are sticky on the ctx;
 *   - one ctx = one GPU = one caller thread at a time (the reference is single-threaded GL:
 *     RayTracing/src/rayTracing.cpp:1229);
 *   - the wire structs are the reference's own structs, byte for byte
 *     (RayTracing/Assets/headers/mesh.h:26-47,112-126; camera.h:10-36), so a maintainer can pass
 *     `rtxTriangles.data()`, `materials.data()` and `&uniforms` unchanged;
 *   - there is NO CPU fallback: without a CUDA device rt_create fails with RT_ERR_NO_DEVICE.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- status codes */
enum {
    RT_OK = 0,
    RT_ERR_INVALID = 1,     /* bad argument / call order                         */
    RT_ERR_NO_DEVICE = 2,   /* no CUDA device (there is no CPU fallback)         */
    RT_ERR_CUDA = 3,        /* a CUDA runtime call or kernel failed (sticky)     */
    RT_ERR_NCCL = 4,        /* NCCL missing or a collective failed (sticky)      */
    RT_ERR_OOM = 5,
    RT_ERR_STATE = 6        /* scene not built, comm not initialised, ...        */
};

/* ---------------------------------------------------------------- material types
 * compute.glsl:7-13 == mesh.h:16-22 */
enum {
    RT_MAT_DIFFUSE = 0,
    RT_MAT_SPECULAR = 1,
    RT_MAT_LIGHT = 2,
    RT_MAT_CHECKER = 3,
    RT_MAT_GLASS = 4,
    RT_MAT_TEXTURE = 5,
    RT_MAT_GLASS_HIGHLIGHT = 6
};
#define RT_MAX_TEXTURES 5 /* compute.glsl:108, mesh.h:24 */

/* ---------------------------------------------------------------- wire structs
 * RTXTriangle, mesh.h:112-126 == `struct Triangle` std430, compute.glsl:46-56.  80 bytes. */
typedef struct rt_triangle {
    float a[4];            /*  0  vec3 in a vec4 slot, w = 0 */
    float b[4];            /* 16 */
    float c[4];            /* 32 */
    float aTex[2];         /* 48  NB: (aTex,bTex,cTex) = (vt1,vt2,vt0), mesh.h:602-606 */
    float bTex[2];         /* 56 */
    float cTex[2];         /* 64 */
    int32_t materialIndex; /* 72 */
    float pad;             /* 76 */
} rt_triangle;

/* Material, mesh.h:26-47 == compute.glsl:17-37.  96 bytes. */
typedef struct rt_material {
    float color[4];            /*  0 */
    float specularColor[4];    /* 16 */
    float emissionColor[4];    /* 32 */
    int32_t textureIndex;      /* 48 */
    float emissionStrength;    /* 52 */
    float smoothness;          /* 56 */
    float specularProbability; /* 60 */
    float checkerScale;        /* 64 */
    float refractiveIndex;     /* 68 */
    int32_t materialType;      /* 72 */
    int32_t index;             /* 76 */
    int32_t isEdgeHighlight;   /* 80 */
    int32_t pad1, pad2, pad3;  /* 84..95 */
} rt_material;

/* GlobalUniforms, camera.h:10-36 == GlobalUniformsBlock std140, compute.glsl:119-146.  192 bytes. */
typedef struct rt_uniforms {
    int32_t pad;                        /*   0 */
    int32_t numTextures;                /*   4 */
    uint32_t width;                     /*   8 */
    uint32_t height;                    /*  12 */
    int32_t numSpheres;                 /*  16  always 0 (rayTracing.cpp:1389) */
    int32_t numTriangles;               /*  20 */
    int32_t basicShading;               /*  24  1 = preview path traceBasic (compute.glsl:565) */
    int32_t basicShadingShadow;         /*  28 */
    float basicShadingLightPosition[4]; /*  32 */
    int32_t environmentalLight;         /*  48 */
    int32_t maxBounceCount;             /*  52 */
    int32_t numRaysPerPixel;            /*  56 */
    uint32_t frameIndex;                /*  60  the reference's only seed input (compute.glsl:668) */
    float cameraPos[4];                 /*  64 */
    float viewportRight[4];             /*  80 */
    float viewportUp[4];                /*  96 */
    float viewportFront[4];             /* 112 */
    float pixelRight[4];                /* 128 */
    float pixelUp[4];                   /* 144 */
    float defocusDiskRight[4];          /* 160 */
    float defocusDiskUp[4];             /* 176 */
} rt_uniforms;

/* Node, BVH.h:54-65 == compute.glsl:58-73.  48 bytes.  NOT consumed by the backend (the GPU builds
 * its own BVH); declared here because the oracle and the reference harness exchange it. */
typedef struct rt_ref_node {
    float bmin[3];
    float pad0;
    float bmax[3];
    float pad1;
    int32_t triangleIndex;
    int32_t triangleCount;
    int32_t childIndex; /* -1 = leaf; children at childIndex, childIndex+1 */
    int32_t pad2;
} rt_ref_node;

/* ---------------------------------------------------------------- configuration */
enum {
    RT_RNG_REF_PCG = 0, /* the reference's sequential hash stream (compute.glsl:148-154,668):
                           one state per pixel, carried across the samples of a frame           */
    RT_RNG_PHILOX = 1   /* counter-based Philox4x32-10 keyed (pixel, frame, sample, bounce, draw):
                           the value of every draw is independent of launch order               */
};
enum {
    RT_SPLIT_NONE = 0,
    RT_SPLIT_TILES = 1, /* image-tile split: this rank renders the row bands it owns, all frames */
    RT_SPLIT_FRAMES = 2 /* frame-slice split: this rank renders frames f with f % world == rank  */
};
enum {
    RT_FIRST_HIT_CENTRE = 0, /* primary ray of traceBasic (compute.glsl:674-676), no RNG         */
    RT_FIRST_HIT_SAMPLE0 = 1 /* jittered sample 0 of frame uniforms.frameIndex (compute.glsl:686-689) */
};

typedef struct rt_config {
    int32_t device;         /* CUDA device ordinal                                               */
    int32_t rng_mode;       /* RT_RNG_*                                                          */
    int32_t split_mode;     /* RT_SPLIT_*                                                        */
    int32_t rank;           /* 0 <= rank < world_size                                            */
    int32_t world_size;     /* 1 = single GPU                                                    */
    int32_t band_rows;      /* RT_SPLIT_TILES: rows per band, bands dealt round-robin; 0 = 8     */
    int32_t instrument;     /* 1 = count node visits / triangle tests per segment (slower build
                               of the same kernels; never used for timed runs)                   */
    int32_t kernel_timing;  /* 1 = bracket every kernel with CUDA events on the ctx stream and report
                               per-class device time through rt_get_counters (small overhead)    */
    uint64_t max_paths_in_flight; /* path slots kept resident (128 B each); 0 = auto: 512 Mi slots,
                                     capped at 40 % of the free device memory                       */
} rt_config;

typedef struct rt_counters {
    uint64_t segments;      /* closest-hit queries traced (primary + bounces) since last reset   */
    uint64_t paths;         /* camera paths started                                              */
    uint64_t node_visits;   /* instrument=1 only: inner nodes fetched                            */
    uint64_t tri_tests;     /* instrument=1 only: triangles tested                               */
    uint64_t extend_launches;
    uint64_t kernel_launches;  /* every kernel of this library launched since last reset         */
    double extend_ms;       /* device time inside k_extend (CUDA events on the ctx stream)       */
    double shade_ms;        /* device time inside raygen/shade/accumulate/resolve                */
    double build_ms;        /* device time of the last rt_scene_build                            */
    uint64_t bvh_nodes;     /* nodes k_extend walks (4-wide)                                       */
    uint64_t bvh_bytes;     /* bytes of node + triangle arrays traversal reads                   */
    uint64_t bvh_depth;     /* longest leaf-to-root path of the GPU BVH                          */
    uint64_t bvh_width;     /* 4 = k_extend walks the 4-wide nodes, 2 = the binary nodes        */
    uint64_t bvh_stack_need;/* worst-case traversal-stack entries of that tree (must be < 256)   */
    uint64_t bvh_build_rounds; /* clustering rounds of the last build (PLOC), 0 for the Karras tree */
    uint64_t extend_blocks_per_sm; /* resident 128-thread blocks of the traversal kernel per SM      */
} rt_counters;

/* Host view of the GPU-built BVH, for validation only (tests check that every triangle lies in
 * its leaf box and that the root box is the scene box).  64-byte inner node, both child boxes in
 * the parent.  child < 0 encodes a leaf: first = ~child, i.e. sorted triangle slot. */
typedef struct rt_bvh_node {
    float lo_x[2], hi_x[2]; /* [0]=left child box, [1]=right child box */
    float lo_y[2], hi_y[2];
    float lo_z[2], hi_z[2];
    int32_t child[2];
    int32_t count[2];       /* triangles under a leaf child (>=1); 0 for an inner child */
} rt_bvh_node;

typedef struct rt_ctx rt_ctx;

/* ---------------------------------------------------------------- lifetime
 * Replaces GL context + object creation / .Delete() (rayTracing.cpp:1215-1242, :1421-1432). */
int rt_create(rt_ctx** out, const rt_config* cfg);
void rt_destroy(rt_ctx* ctx);
const char* rt_last_error(const rt_ctx* ctx); /* owned by ctx; "" if none. ctx may be NULL → static text */
const char* rt_version(void);

/* Launch on the caller's CUDA stream (a cudaStream_t passed as void*).  NULL = the ctx's own
 * non-blocking stream.  Lets a host time the library with its own events. */
int rt_set_stream(rt_ctx* ctx, void* cuda_stream);

/* ---------------------------------------------------------------- scene upload
 * Replaces `SSBO trianglesSSBO(rtxTriangles.data(), 80*n, 1)` and
 * `SSBO materialsSSBO(materials.data(), 96*k, 3)` (rayTracing.cpp:1323-1325; SSBO.cpp:3-10):
 * the library copies, the caller keeps ownership and may free at once.  Triangles are passed in the
 * caller's ORIGINAL order (before any BVH permutation); triangle ids reported by this library are
 * indices into that array. */
int rt_scene_set_triangles(rt_ctx* ctx, const rt_triangle* tris, int64_t count);
int rt_scene_set_materials(rt_ctx* ctx, const rt_material* mats, int32_t count);

/* Replaces `Texture2D(path, GL_TEXTURE0+i)` (mesh.h:310-318; textureClass.cpp:55-114) and the
 * sampler binding (rayTracing.cpp:1315-1320).  `pixels` = what stbi_load returned AFTER
 * stbi_set_flip_vertically_on_load(true): row 0 is the bottom row, 8-bit, `channels` in 1..4.
 * Sampling semantics kept: bilinear, REPEAT, no mips, no sRGB decode, 1 channel → (r,r,r). */
int rt_scene_set_texture(rt_ctx* ctx, int32_t slot, const uint8_t* pixels, int32_t width,
                         int32_t height, int32_t channels);

/* Replaces `BVH BVH(bvhTriangles, rtxTriangles)` (rayTracing.cpp:1293; BVH.h:150-220) and the node
 * SSBO upload (rayTracing.cpp:1324): builds a BVH on the GPU (Morton codes, radix sort, PLOC
 * clustering — or the Karras LBVH with RT_BVH_BUILDER=lbvh — then 32-byte quantised binary nodes and their
 * collapse into 64-byte 4-wide nodes) and re-lays the triangles out for traversal. */
int rt_scene_build(rt_ctx* ctx);

/* ---------------------------------------------------------------- render
 * Replaces `UBO.Update(&uniforms,192)` + `glDispatchCompute(W/8,H/4,1)` + barrier
 * (rayTracing.cpp:188-192, :1402-1406): one frame of uniforms->numRaysPerPixel samples per pixel
 * (or the traceBasic preview when uniforms->basicShading != 0) into the RGBA32F image.
 * Asynchronous; uniforms are read before the call returns. */
int rt_render_frame(rt_ctx* ctx, const rt_uniforms* uniforms);

/* Replaces reading image binding 0 (compute.glsl:5,700): W*H*4 floats, row 0 = bottom row.
 * Blocking (mirrors glReadPixels).  With RT_SPLIT_TILES only the rows this rank owns are defined. */
int rt_read_frame_rgba32f(rt_ctx* ctx, float* dst);

/* Replaces screenshot() (rayTracing.cpp:124-283, the frame loop :184-242, average :248-250,
 * flip :253-259): renders `frames` frames with frameIndex = 0..frames-1, quantises each frame to
 * 8 bit after ACES + gamma, sums, divides by `frames`, truncates, flips to top-down RGB8.
 * Multi-GPU: the partial sums are reduced / gathered to rank 0 over NCCL; only rank 0 writes
 * `rgb8_topdown` (W*H*3 bytes; may be NULL on other ranks).  Blocking. */
int rt_screenshot(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames, uint8_t* rgb8_topdown);

/* Same work as rt_screenshot but the result stays in device memory (no D2H): used to measure the
 * device-resident throughput.  rt_screenshot_fetch copies the last result out. */
int rt_screenshot_device(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames);
int rt_screenshot_fetch(rt_ctx* ctx, uint8_t* rgb8_topdown);

/* The multi-GPU pieces of rt_screenshot, exposed so that ranks can also be emulated one after the
 * other on a single GPU: render this rank's share into the 8-bit frame sums (W*H*3 u32, row 0 =
 * bottom, zero where the rank owns nothing), read them, and finalise any summed buffer
 * (rayTracing.cpp:248-259). */
int rt_screenshot_partial(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t frames);
int rt_read_frame_sum(rt_ctx* ctx, uint32_t* sums_bottom_up);
int rt_finalize_sums(rt_ctx* ctx, const uint32_t* sums_bottom_up, int32_t width, int32_t height,
                     int32_t frames, uint8_t* rgb8_topdown);

/* ---------------------------------------------------------------- parity hooks
 * Host-memory entry points that return when their results are in the caller's arrays.  Both are the closest-hit
 * query (rt_query_closest with no tmax) run on device copies of the rays, so they report exactly what it reports. */
/* Closest hit of the primary ray of every pixel: tri_id[y*W+x] = index into the array given to
 * rt_scene_set_triangles, or -1 for a miss; dst = hit distance (1e38f for a miss).  Row 0 = bottom.
 * Ties in dst are broken by the lowest triangle index. */
int rt_first_hit(rt_ctx* ctx, const rt_uniforms* uniforms, int32_t mode, int32_t* tri_id,
                 float* dst);

/* Closest hit of `count` caller-supplied rays (origins/dirs: count*3 floats).  Outputs may be NULL. */
int rt_trace_rays(rt_ctx* ctx, const float* origins, const float* dirs, int64_t count,
                  int32_t* tri_id, float* dst, float* bary_u, float* bary_v);

/* ---------------------------------------------------------------- ray queries on device memory
 * Ray queries on DEVICE memory, asynchronous on the ctx stream (rt_set_stream): no host synchronisation and no device
 * allocation once the scene is built.  origins / dirs: count*3 floats; tmax: count floats or NULL (unbounded).
 * A hit needs 1e-6 < t < min(tmax, 1e38); a NaN, zero or negative tmax never hits.  Every pointer must be device
 * (or managed) memory of cfg.device, else RT_ERR_INVALID; so are count < 0 and count > 2^30, both rejected before
 * anything is enqueued.  count == 0 returns RT_OK and launches nothing; an unbuilt scene returns RT_ERR_STATE.
 * The ray count and work cursor are device words of the ctx, so two queries on one ctx are ordered by the ctx
 * stream, as every other call is: the caller orders the stream against the producers of the inputs and the consumers
 * of the outputs (e.g. with events).
 *
 * rt_query_closest: the closest hit, exactly what rt_trace_rays reports for the same ray when its distance is below
 * tmax, and a miss otherwise.  tri_id indexes the array given to rt_scene_set_triangles, exact ties go to the lowest
 * id; a miss writes -1 / 1e38 / 0 / 0.  Outputs may be NULL (not written); they are written in stream order. */
int rt_query_closest(rt_ctx* ctx, const float* origins, const float* dirs, const float* tmax, int64_t count,
                     int32_t* tri_id, float* dst, float* bary_u, float* bary_v);
/* rt_query_occluded: occluded[i] = 1 if some triangle is hit with t < tmax[i], else 0 (the same as
 * rt_query_closest's dst < tmax, but the walk stops at the first such triangle).  occluded must not be NULL. */
int rt_query_occluded(rt_ctx* ctx, const float* origins, const float* dirs, const float* tmax, int64_t count,
                      uint8_t* occluded);

/* ---------------------------------------------------------------- nearest-triangle queries on device memory
 * For each point p (points: count*3 floats) and radius r = max_dist[i] (max_dist: count floats, or NULL = unbounded):
 * among the triangles T with dist(p, T) < min(r, 1e38), the one with the smallest distance to the CLOSED triangle
 * (interior, edges, vertices; a distance of 0 is a hit); exact ties go to the lowest id.  Outputs per point: tri_id
 * (index into the array given to rt_scene_set_triangles), dist, bary_u / bary_v with closest point a + (b-a) u +
 * (c-a) v, and that point (closest: count*3 floats).  A miss writes -1 / 1e38 / 0 / 0 and (0, 0, 0).  A NaN, zero
 * or negative radius and a point with a non-finite coordinate never hit.  A distance whose square overflows binary32
 * (beyond about 1.8e19) is +inf and never hits.  The point-triangle distance is defined, bit for bit, by the CPU
 * oracle (DESIGN.md §5).  Sorting the points for spatial coherence is left to the caller.
 * Same rules as the ray queries: asynchronous on the ctx stream, every non-NULL pointer must be device (or managed)
 * memory of cfg.device and points must not be NULL, else RT_ERR_INVALID, as are count < 0 and count > 2^30, all
 * rejected before anything is enqueued; count == 0 returns RT_OK and launches nothing; an unbuilt scene returns
 * RT_ERR_STATE.  Outputs may be NULL (not written). */
int rt_query_nearest(rt_ctx* ctx, const float* points, const float* max_dist, int64_t count, int32_t* tri_id,
                     float* dist, float* bary_u, float* bary_v, float* closest);

/* Export the GPU-built BVH: call with nodes == NULL to get sizes.  sorted_tri_ids[slot] = original
 * triangle index stored at that leaf slot. */
int rt_scene_get_bvh(rt_ctx* ctx, rt_bvh_node* nodes, int64_t* node_count, int32_t* sorted_tri_ids,
                     int64_t* tri_count, float scene_lo[3], float scene_hi[3]);

int rt_get_counters(rt_ctx* ctx, rt_counters* out);
int rt_reset_counters(rt_ctx* ctx);

/* ---------------------------------------------------------------- multi-GPU (one process per GPU)
 * NCCL is loaded with dlopen("libnccl.so.2") on first use, so a process that already carries NCCL
 * (e.g. through torch) shares that copy.  Rank 0 makes the id, the host broadcasts the 128 bytes by
 * any means (torch.distributed, MPI, a file), every rank calls rt_comm_init. */
int rt_comm_unique_id(uint8_t id_out[128]);
int rt_comm_init(rt_ctx* ctx, const uint8_t id[128]);

/* Which rows does `rank` own under RT_SPLIT_TILES?  Pure host arithmetic (no GPU needed):
 * writes up to `cap` row indices, returns the number of rows owned. */
int64_t rt_split_rows(int32_t height, int32_t band_rows, int32_t rank, int32_t world_size,
                      int32_t* rows_out, int64_t cap);
/* Which frames does `rank` own under RT_SPLIT_FRAMES? */
int64_t rt_split_frames(int32_t frames, int32_t rank, int32_t world_size, int32_t* frames_out,
                        int64_t cap);
/* How rt_screenshot cuts `frames` frames of `samples_per_pixel` samples over `local_pixels` pixels into wavefront
 * batches under a budget of `max_paths_in_flight` path slots (the loop nest that replaces the reference's
 * per-frame dispatch, rayTracing.cpp:184-192): samples of one frame in flight together, and how many frames
 * share a batch.  Pure host arithmetic, no GPU needed; it never changes a bit of the output. */
int rt_plan_batches(uint64_t max_paths_in_flight, int64_t local_pixels, int32_t samples_per_pixel, int32_t frames,
                    int32_t rng_mode, int32_t* samples_per_batch, int32_t* frames_per_batch);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
