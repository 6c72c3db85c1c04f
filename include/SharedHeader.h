/* SharedHeader.h -- the host/device shared records of the ray-cast + radiance path.
 *
 * The reference's test/SharedHeader.h:1-3 is an empty shim; the records it was
 * meant to hold are declared twice there: on the host in
 * test/RaytraceTest.cpp:50-76 (#pragma pack(1), 64 B each) and again in
 * test/ClKernels/GenerateColors.cl:12-28.  This header is the single definition
 * for this repo: byte-identical 64-byte Triangle / Material records (the API
 * format a caller uploads), plus the B200-side records the BVH path uses
 * (64-byte two-child node, 48-byte precomputed-edge triangle) and the render
 * parameter block that replaces the reference's hard-coded constants.
 *
 * Plain C (C99) and C++ compatible; no CUDA or torch types.
 */
#ifndef PTB200_SHARED_HEADER_H
#define PTB200_SHARED_HEADER_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTB_DIFFUSE 1  /* GenerateColors.cl:3 */
#define PTB_SPECULAR 2 /* GenerateColors.cl:4 */

typedef struct ptb_float4 {
    float x, y, z, w;
} ptb_float4;

/* RaytraceTest.cpp:9-15 -- the by-value kernel constant {W, H, frame, unused} */
typedef struct ptb_int4 {
    int32_t x, y, z, w;
} ptb_int4;

/* RaytraceTest.cpp:50-59 / GenerateColors.cl:12-19.  Indexed by QUAD id. */
typedef struct ptb_material {
    ptb_float4 albedo;   /* 16 */
    ptb_float4 emissive; /* 16 */
    float roughness;     /* 4  (GGX alpha, used as-is) */
    int32_t type;        /* 4  PTB_DIFFUSE | PTB_SPECULAR */
    char padding[24];
} ptb_material;

/* RaytraceTest.cpp:61-76 / GenerateColors.cl:21-28.  id = quad id. */
typedef struct ptb_triangle {
    ptb_float4 p1; /* 16, w = 0 */
    ptb_float4 p2; /* 16 */
    ptb_float4 p3; /* 16 */
    int32_t id;    /* 4 */
    char padding[12];
} ptb_triangle;

/* ---- B200-side records (BUILD-DEFINED; the reference has no BVH) ---------- */

/* BVH nodes hold the (padded) boxes of their CHILDREN, so one coalesced fetch decides every descent from
 * that node.  Boxes are stored as CENTRE and HALF-EXTENT (box = [c - e, c + e]): the slab test is then three
 * FMAs per axis and needs no per-axis min/max (t_centre = c*invd - o*invd, t_near = t_centre - e*|invd|,
 * t_far = t_centre + e*|invd|).  Child reference: >= 0 internal node index; < 0 leaf, decoded as
 * first = (~ref) >> 3, count = ((~ref) & 7) + 1 into the ordered triangle array; PTB_BVH_EMPTY = unused slot
 * (its box has e = -1e30 and never hits).
 *
 * Two node widths (and the FLAT form below), chosen per scene (DESIGN.md section 3):
 *   ptb_bvh_node   binary, 4 x 128-bit words = 64 B  -- scenes traversed from L2/HBM (fewest bytes and registers
 *                                                        per visit; measured best on the 2M-triangle scene)
 *   ptb_bvh_node4  4-wide, 8 x 128-bit words = 128 B -- scenes that live entirely in shared memory (half as many
 *                                                        loop iterations per ray; measured +8 % on Cornell AO)   */
typedef struct ptb_bvh_node {
    float c0[3];
    int32_t child0; /* word 0: child-0 centre,      child-0 ref */
    float e0[3];
    int32_t child1; /* word 1: child-0 half-extent, child-1 ref */
    float c1[3];
    int32_t pad0; /* word 2: child-1 centre */
    float e1[3];
    int32_t pad1; /* word 3: child-1 half-extent */
} ptb_bvh_node;

/* Quantised encoding of a binary node, 2 x 128-bit words = 32 B: what the kernels traverse for width-2 scenes (one 256-bit load
 * per visit instead of two: the L1 data pipe, one wavefront per clock and SM, is what binds the traversal of a scene that lives in
 * L2/HBM).  Box planes are 16-bit indices on a grid over the scene: plane = grid_lo[axis] + q * grid_step[axis].  The encoding is a
 * pure function of the ptb_bvh_node array (rules Q1-Q3, csrc/lbvh.cuh: k_quant_grid / k_quant_nodes == the CPU oracle's
 * ora_bvh_quantize): every quantised box contains its fp32 box with a full grid step to spare.  Node numbering = ptb_bvh_node's. */
typedef struct ptb_bvh_nodeq {
    uint32_t box0[3]; /* child 0: x, y, z words, each lo plane | hi plane << 16 */
    uint32_t box1[3]; /* child 1 */
    int32_t child0, child1;
} ptb_bvh_nodeq;

typedef struct ptb_bvh_node4 {
    float c0[3];
    int32_t child0; /* word 0: child-0 centre,      child-0 ref */
    float e0[3];
    int32_t child1; /* word 1: child-0 half-extent, child-1 ref */
    float c1[3];
    int32_t child2; /* word 2: child-1 centre,      child-2 ref */
    float e1[3];
    int32_t child3; /* word 3: child-1 half-extent, child-3 ref */
    float c2[3];
    int32_t pad0;
    float e2[3];
    int32_t pad1;
    float c3[3];
    int32_t pad2;
    float e3[3];
    int32_t pad3;
} ptb_bvh_node4;

/* FLAT form for scenes of <= PTB_FLAT_MAX_LEAVES leaves and <= 64 triangles (the Cornell box: 18 leaves, 36 triangles):
 * no tree at all -- the leaf slots of the binary tree in leaf order, each with its padded box (centre / half-extent, as
 * above) and the 64-bit mask of the positions its triangles occupy in the ordered triangle array.  A query slab-tests
 * EVERY leaf box in straight-line code (all 32 lanes of a warp busy, the records are kernel parameters read as
 * constant-bank operands), ORs the masks of the boxes it hits, then runs Moller-Trumbore over the set bits.  There is no
 * stack, no child ordering and no trip-count divergence in the box phase (DESIGN.md section 3).            */
typedef struct ptb_bvh_leafbox {
    float c[3];
    uint32_t mask_lo; /* word 0: box centre,      triangle positions 0..31 of this leaf */
    float e[3];
    uint32_t mask_hi; /* word 1: box half-extent, triangle positions 32..63 */
} ptb_bvh_leafbox;
#define PTB_FLAT_MAX_LEAVES 32
#define PTB_FLAT_MAX_TRIS 64

#define PTB_BVH_WIDTH 4
#define PTB_MAX_PEERS 7 /* peer images a gathering render can store into (8 GPUs per node) */ /* slots of a ptb_bvh_node4 */
#define PTB_BVH_EMPTY 0x7fffffff
#define PTB_BVH_LEAF_REF(first, count) (~(int32_t)(((uint32_t)(first) << 3) | (uint32_t)((count)-1)))
#define PTB_BVH_LEAF_FIRST(ref) ((int32_t)((uint32_t)(~(ref)) >> 3))
#define PTB_BVH_LEAF_COUNT(ref) ((int32_t)(((uint32_t)(~(ref))) & 7u) + 1)
#define PTB_BVH_MAX_LEAF 8

/* Triangle in BVH order, precomputed-edge layout: e1 = p2 - p1 and e2 = p3 - p1
 * are the very fp32 subtractions GenerateColors.cl:92-93 performs per test, only
 * hoisted, so Moller-Trumbore stays bit-identical.  3 x 128-bit words.         */
typedef struct ptb_bvh_tri {
    float p1[3];
    int32_t index; /* position in the caller's Triangle array (tie-break key) */
    float e1[3];
    int32_t quad; /* Triangle.id */
    float e2[3];
    int32_t pad;
} ptb_bvh_tri;

/* ---- render parameters ---------------------------------------------------- */

enum {
    PTB_MODE_PRIMARY = 0, /* C1: primary ray, hit-ID outputs                          */
    PTB_MODE_AO = 1,      /* C2: primary + ao_samples cosine-hemisphere any-hit rays   */
    PTB_MODE_DIRECT = 2,  /* C3: primary + 1 shadow ray to the area light             */
    PTB_MODE_PATH = 3     /* C4/C5: GenerateColors.cl:223-261 traceRays                */
};
enum {
    PTB_ACCUM_REFERENCE = 0, /* GenerateColors.cl:314-321 gamma-space running mean      */
    PTB_ACCUM_LINEAR = 1     /* fp32 sum in frame order, divided by n_frames at resolve */
};
enum { PTB_INTEGRATOR_AUTO = 0, PTB_INTEGRATOR_MEGAKERNEL = 1, PTB_INTEGRATOR_WAVEFRONT = 2 };
enum { PTB_ACCEL_BVH = 0, PTB_ACCEL_BRUTE = 1 };
enum {
    PTB_OUTPUT_FLOAT4 = 0, /* the reference's framebuffer: float4 per pixel                                   */
    PTB_OUTPUT_RGB8 = 1    /* the reference's final output transform done on the device: sqrt, x255, truncate,
                              clamp (RaytraceTest.cpp:78-83,:283) -> 3 bytes per pixel, the PPM payload      */
};

/* Defaults (ptb_render_params_default) equal the reference's hard-coded values:
 * 512x512 (RaytraceTest.cpp:219), BOUNCES 16 (GenerateColors.cl:5), frame
 * protocol RaytraceTest.cpp:250-253.                                          */
typedef struct ptb_render_params {
    int32_t width, height;
    int32_t first_frame, n_frames; /* frames first_frame .. first_frame+n_frames-1 */
    int32_t mode;                  /* PTB_MODE_*        */
    int32_t accum;                 /* PTB_ACCUM_*       */
    int32_t integrator;            /* PTB_INTEGRATOR_*  */
    int32_t accel;                 /* PTB_ACCEL_*       */
    int32_t max_depth;             /* path segments, reference 16 */
    int32_t ao_samples;            /* AO rays per primary hit, C2: 16 */
    float ao_max_dist;             /* AO any-hit tmax */
    int32_t light_quad;            /* quad id of the area light (cornellbox: 5) */
    /* area-light parallelogram P = p1 + xi1*ea + xi2*eb; all-zero ea = derive it
     * from the first triangle pair whose id is light_quad                        */
    float light_p1[3], light_ea[3], light_eb[3];
    /* image sharding: this call renders the pixels gid with
     * (gid / shard_block) % shard_count == shard_index; outputs are compacted
     * to local index (gid / (shard_block*shard_count))*shard_block + gid % shard_block */
    int32_t shard_index, shard_count, shard_block;
    int32_t collect_stats; /* 1: fill per-pixel hit-ID / visit outputs and counters */
    int32_t frames_per_batch; /* wavefront: samples kept in flight; 0 = auto */
    int32_t output;           /* PTB_OUTPUT_*: what ptb_render_host / _async copy to the host (device entry points always
                                 keep the float4 frame); RGB8 needs accum LINEAR or first_frame 0                       */
    int32_t reserved[6];
} ptb_render_params;

/* Ray/test counters (exact integers).  Rays = scene queries (closest or any).
 * Stage counters feed SURVEY.md 8(d)'s flops/bytes-per-ray formula.           */
typedef struct ptb_counters {
    uint64_t rays_closest; /* closest-hit queries */
    uint64_t rays_any;     /* any-hit (shadow / AO) queries */
    uint64_t nodes;        /* internal BVH node records fetched (2 or 4 slab tests each) */
    uint64_t tri_tests;    /* Moller-Trumbore tests started (det stage) */
    uint64_t samples;      /* pixel-frames */
    uint64_t reserved[3];
} ptb_counters;

/* ---- scene queries on caller-owned device ray buffers (ptb_scene_intersect) -------------------
 * One ray = 32 bytes, read with one 256-bit load (the array must be 32-byte aligned).  A query accepts a triangle at
 * 0 < t < tmax (tmax <= 0 or NaN: a miss); there is no tmin, so callers offset their origins (the reference uses
 * p + 0.01 * wi).  One hit = 16 bytes: tri = index into the caller's triangle array or -1 (then t = u = v = 0); the
 * quad id of a hit is tris[tri].id.                                                                             */
typedef struct ptb_ray {
    float o[3];
    float tmax;
    float d[3];
    int32_t reserved;
} ptb_ray;
typedef struct ptb_hit {
    float t, u, v;
    int32_t tri;
} ptb_hit;
enum {
    PTB_QUERY_CLOSEST = 0, /* smallest t; equal t -> lowest caller index                  */
    PTB_QUERY_ANY = 1      /* the first triangle accepted in traversal order (shadow rays) */
};

/* ---- render-mode samples along caller-owned device rays (ptb_scene_shade) -------------------------------------------
 * One sample = 32 bytes, read with one 256-bit load (the array must be 32-byte aligned).  seed is the RNG state of the sample
 * (GenerateColors.cl:47-71) after whatever draws the caller's camera made: the reference's camera starts from
 * gid + hash_uint32(frame) (:308) and draws two floats for its jitter (:278-279).  d need not be normalised; the render
 * modes use it as given.                                                                                               */
typedef struct ptb_sample_ray {
    float o[3];
    uint32_t seed;
    float d[3];
    int32_t reserved; /* ignored */
} ptb_sample_ray;

#ifdef __cplusplus
} /* extern "C" */
#if __cplusplus >= 201103L
static_assert(sizeof(ptb_ray) == 32, "ray record must be 32 bytes (one 256-bit load)");
static_assert(sizeof(ptb_hit) == 16, "hit record must be 16 bytes (one 128-bit store)");
static_assert(sizeof(ptb_sample_ray) == 32, "sample ray record must be 32 bytes (one 256-bit load)");
static_assert(sizeof(ptb_material) == 64, "Material must be 64 bytes (RaytraceTest.cpp:50-59)");
static_assert(sizeof(ptb_triangle) == 64, "Triangle must be 64 bytes (RaytraceTest.cpp:61-76)");
static_assert(sizeof(ptb_bvh_node) == 64, "binary BVH node must be 64 bytes");
static_assert(sizeof(ptb_bvh_nodeq) == 32, "quantised binary BVH node must be 32 bytes");
static_assert(sizeof(ptb_bvh_node4) == 128, "4-wide BVH node must be 128 bytes");
static_assert(sizeof(ptb_bvh_tri) == 48, "BVH triangle must be 48 bytes");
static_assert(sizeof(ptb_bvh_leafbox) == 32, "flat leaf box must be 32 bytes");
#endif
#endif

#endif /* PTB200_SHARED_HEADER_H */
