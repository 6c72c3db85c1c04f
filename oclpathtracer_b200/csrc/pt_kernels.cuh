// pt_kernels.cuh -- sm_100a kernels of the ray-cast + radiance path.
//
//   k_mega<MODE,...>   one thread = one sample (pixel x frame): camera ray, scene
//                      queries and shading in registers; scene staged in shared
//                      memory by one TMA bulk copy per CTA.
//   k_resolve          ordered per-pixel accumulation of a batch of samples
//                      (GenerateColors.cl:314-321 or linear mean).
//   k_trace            scene queries on caller-supplied rays (parity tests).
//   wavefront stages   pt_wavefront.cuh
#pragma once

#include "pt_device.cuh"

namespace ptd {

// ---- counters ---------------------------------------------------------------------------
enum { CTR_CLOSEST = 0, CTR_ANY = 1, CTR_NODES = 2, CTR_TESTS = 3, CTR_SAMPLES = 4, CTR_COUNT = 8 };

PTD_FI void flush_counter(unsigned long long* counters, int which, uint32_t v) {
    const uint32_t total = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && total) atomicAdd(&counters[which], (unsigned long long)total);
}

// ---- shared-memory staging with the bulk async-copy engine (TMA, 1-D) -------------------
//
// layout (16-byte aligned pieces):  [mbarrier 16 B][nodes][triangles][materials][stack_ref][stack_tn]

PTD_FI uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

PTD_FI void bulk_g2s(void* dst, const void* src, uint32_t bytes, void* mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(mbar))
                 : "memory");
}

// NODES: stage the node prefix and carve the traversal stack; TRIS_BVH: triangle
// positions refer to the BVH-ordered array (else the caller-ordered one).
template <bool NODES, int SMALL, bool TRIS_BVH = NODES>
PTD_FI Ctx stage_scene(const SceneDev& sc, unsigned char* smem) {
    constexpr bool BVH = NODES;
    constexpr bool STACK = NODES && SMALL != PTD_FLAT;  // FLAT scenes need no traversal stack
    Ctx c;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem);
    unsigned char* p = smem + 16;
    const uint32_t node_bytes = !BVH ? 0u : SMALL == PTD_FLAT ? (uint32_t)sc.flat_n * 32u : (uint32_t)sc.smem_nodes * (SMALL ? 128u : 32u);
    const uint32_t tri_bytes = SMALL ? (uint32_t)sc.n_tris * 48u : 0u;
    const uint32_t mat_bytes = SMALL ? (uint32_t)sc.n_mats * 32u : 0u;
    float4* s_nodes = reinterpret_cast<float4*>(p);
    float4* s_tris = reinterpret_cast<float4*>(p + node_bytes);
    float4* s_mats = reinterpret_cast<float4*>(p + node_bytes + tri_bytes);
    unsigned char* s_stack = p + node_bytes + tri_bytes + mat_bytes;

    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(mbar)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t total = node_bytes + tri_bytes + mat_bytes;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(total)
                     : "memory");
        if (node_bytes) bulk_g2s(s_nodes, sc.nodes, node_bytes, mbar);
        if (tri_bytes) bulk_g2s(s_tris, TRIS_BVH ? sc.tris : sc.tris_orig, tri_bytes, mbar);
        if (mat_bytes) bulk_g2s(s_mats, sc.mats, mat_bytes, mbar);
    }
    // every thread waits for phase 0 to complete (bytes landed)
    {
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n"
                "selp.u32 %0, 1, 0, p;\n"
                "}\n"
                : "=r"(done)
                : "r"(smem_u32(mbar))
                : "memory");
        }
    }
    c.s_nodes = smem_u32(s_nodes);
    c.s_tris = smem_u32(s_tris);
    c.s_mats = smem_u32(s_mats);
    c.g_nodes = sc.nodes;
    c.g_tris = TRIS_BVH ? sc.tris : sc.tris_orig;
    c.g_mats = sc.mats;
    c.stride_bytes = blockDim.x * 4u;
    const uint32_t stack_bytes = (STACK && !sc.lstack) ? (uint32_t)sc.stack_depth * blockDim.x * 4u : 0u;
    // two disjoint areas: warps of one CTA can be in a closest-hit and an any-hit query at the same time (AO, DIRECT)
    c.s_stack64 = smem_u32(s_stack) + threadIdx.x * 8u;                       // (ref, entry distance) pairs
    c.s_stack_ref = smem_u32(s_stack) + 2u * stack_bytes + threadIdx.x * 4u;  // any-hit: references only
    c.s_scratch = smem_u32(s_stack) + 3u * stack_bytes + threadIdx.x * 4u;
    c.smem_nodes = sc.smem_nodes;
    c.n_tris = sc.n_tris;
    c.lstack = nullptr;
    c.ld256 = sc.ld256;
    c.flat_n = sc.flat_n;
    for (int k = 0; k < 3; ++k) { c.q_lo[k] = sc.q_lo[k]; c.q_step[k] = sc.q_step[k]; }
    // FLAT scenes have no traversal stack: the area after the staged records is the warps' scratch for flat_mt_coop
    c.s_coop = (BVH && SMALL == PTD_FLAT) ? smem_u32(s_stack) + (threadIdx.x >> 5) * (uint32_t)flat_coop_bytes_per_warp(sc.n_tris) : 0u;
    return c;
}

// host helper: bytes of dynamic shared memory for a launch
static inline size_t scene_smem_bytes(const SceneDev& sc, bool bvh, int small, int block, size_t scratch_per_thread = 0) {
    size_t b = 16;
    if (bvh) b += small == PTD_FLAT ? (size_t)sc.flat_n * 32 : (size_t)sc.smem_nodes * (small ? 128 : 32);
    if (small) b += (size_t)sc.n_tris * 48 + (size_t)sc.n_mats * 32;
    if (bvh && small != PTD_FLAT && !sc.lstack) b += (size_t)sc.stack_depth * block * 12;  // closest-hit pairs (8 B) + any-hit references (4 B)
    if (bvh && small == PTD_FLAT) b += (size_t)(block / 32) * (PTD_COOP_FIXED_BYTES + (((size_t)sc.n_tris * 64 + 15) & ~size_t(15)));  // flat_mt_coop scratch per warp
    return b + scratch_per_thread * block;
}

// ---- per-sample integrators ------------------------------------------------------------------

struct RenderArgs {
    int width, height;
    int first_frame;      // frame index of batch slot 0
    int frames_in_batch;
    int n_local;          // pixels of this shard
    int max_depth, ao_samples;
    float ao_max_dist;
    int light_quad;
    float light_p1[3], light_ea[3], light_eb[3];
    float cam_inv_w, cam_inv_h, cam_aspect;  // CamScale of (width, height), computed by the host
    float light_n[3], light_area;  // normalize(cross(ea, eb)) and |cross(ea, eb)|: the same for every sample, computed once by the host with the same IEEE operations
    Shard shard;
    float4* samples;            // [frames_in_batch][n_local] radiance (xyz)
    ptb_pixel_stats* stats;     // per local pixel, written for stats_frame only
    int stats_frame;
    unsigned long long* counters;
    int tune[16];          // experiment knobs (ptb_device_set_tuning); never change results
};

// Where the sample of a slot gets its ray and its RNG state (template parameter SRC of k_mega, k_mega_path_regen and path_sm2,
// which take their arguments as SRC::Args).
//   CameraRays  ptb_render: slot -> (pixel, frame) -> the reference's camera, GenerateColors.cl:305-310
//   SampleRays  ptb_scene_shade: record `slot` of the caller's ptb_sample_ray array (o, seed, d, unused), one 256-bit load; the
//               sample writes samples[slot] and, with statistics, stats[slot] (frames_in_batch = 1, n_local = the ray count)
struct ShadeArgs : RenderArgs {
    const float4* rays;  // 2 x float4 per ptb_sample_ray record, 32-byte aligned
};
struct CameraRays {
    static constexpr bool buffer = false;
    using Args = RenderArgs;
};
struct SampleRays {
    static constexpr bool buffer = true;
    using Args = ShadeArgs;
};
PTD_FI void load_sample_ray(const ShadeArgs& a, long long slot, Ray& r, uint32_t& seed) {
    float4 o, d;
    ldg256(a.rays + 2 * (size_t)slot, o, d);
    r.o = xyz(o);
    r.d = xyz(d);
    seed = __float_as_uint(o.w);
}

template <bool STATS>
struct SampleStats {
    int tri, quad;
    uint32_t t_bits, visits_primary, visits_secondary, count, id_hash, tri_tests;
};
template <>
struct SampleStats<false> {};

template <bool STATS>
PTD_FI void st_primary(SampleStats<STATS>& st, bool hit, const Hit& h, int quad, uint32_t visits) {
    if constexpr (STATS) {
        st.tri = hit ? h.idx : -1;
        st.quad = hit ? quad : -1;
        st.t_bits = hit ? __float_as_uint(h.t) : 0u;
        st.visits_primary = visits;
    }
}
template <bool STATS>
PTD_FI void st_secondary(SampleStats<STATS>& st, int tri, uint32_t visits) {
    if constexpr (STATS) {
        st.visits_secondary += visits;
        st.id_hash = st.id_hash * 31u + (uint32_t)(tri + 2);
    }
}

struct RayCount {
    uint32_t closest, any;
};

// The path state that the shading step reads and writes: the ray, the RNG state, the radiance and the throughput mask.
// PathRegs keeps it in registers; k_path_sm2 keeps it in shared memory (PathCol) and loads each field where it is used.
struct PathRegs {
    Ray& r;
    uint32_t& seed;
    V3& radiance;
    V3& mask;
    V3 hp;  // the hit point
    PTD_FI V3 o() const { return r.o; }
    PTD_FI V3 d() const { return r.d; }
    PTD_FI uint32_t rng() const { return seed; }
    PTD_FI V3 rad() const { return radiance; }
    PTD_FI V3 msk() const { return mask; }
    PTD_FI V3 hit_point() const { return hp; }
    PTD_FI void set_rng(uint32_t v) { seed = v; }
    PTD_FI void set_rad(V3 v) { radiance = v; }
    PTD_FI void set_msk(V3 v) { mask = v; }
    PTD_FI void set_hit_point(V3 v) { hp = v; }
    PTD_FI void set_ray(const Ray& v) { r = v; }
};

// The part of one path-loop iteration that follows the scene query, GenerateColors.cl:233-257: `hit`/`h` are the query's
// result, `visits` its node visits.  Returns true when the path goes on (ray, mask, seed updated), false when it ended;
// radiance accumulates either way.
template <int SMALL, bool STATS, class PS>
PTD_FI bool path_after_hit(const Ctx& c, bool hit, const Hit& h, PS& ps, int i, int max_depth, SampleStats<STATS>& st,
                           uint32_t visits) {
    V3 p1, e1, e2; int idx = -1, quad = -1;
    if (hit) load_tri<SMALL>(c, h.pos, p1, e1, e2, idx, quad);
    if constexpr (STATS) {
        if (i == 0) st_primary(st, hit, h, quad, visits);
        else st_secondary(st, hit ? h.idx : -1, visits);
        st.count++;
    }
    if (!hit) {  // :233-237, max(bg, 0) = bg
        const V3 radiance = ps.rad(), mask = ps.msk();
        ps.set_rad(mk(radiance.x + mask.x * 0.45f, radiance.y + mask.y * 0.45f, radiance.z + mask.z * 0.45f));
        return false;
    }
    V3 p, n;
    hit_point_normal(e1, e2, ps.o(), ps.d(), h, p, n);
    ps.set_hit_point(p);
    V3 albedo, emissive; float roughness; int type;
    load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);  // :239
    {
        const V3 radiance = ps.rad(), mask = ps.msk();
        ps.set_rad(mk(radiance.x + mask.x * emissive.x * 3.0f, radiance.y + mask.y * emissive.y * 3.0f,
                      radiance.z + mask.z * emissive.z * 3.0f));  // :241
    }
    if (i + 1 >= max_depth) return false;  // the last segment's BSDF sample cannot reach the radiance
    const V3 d = ps.d();
    n = dot(n, d) < 0.0f ? n : mul(n, -1.0f);                     // :243
    V3 wi = mk(0.0f, 0.0f, 0.0f);
    const V3 wo = neg(d);                                         // :246
    float pdf = 0.0f;                                             // :247
    uint32_t seed = ps.rng();
    const V3 color = brdf(wo, wi, pdf, n, albedo, roughness, type, seed);  // :249
    ps.set_rng(seed);
    if (pdf <= 0.0f) return false;                                // :251
    const float dw = dot(wi, n);
    const V3 mask = ps.msk();
    ps.set_msk(mk(mask.x * (color.x * dw / pdf), mask.y * (color.y * dw / pdf), mask.z * (color.z * dw / pdf)));  // :253-255
    ps.set_ray(get_ray(add(ps.hit_point(), mul(wi, 0.01f)), wi));  // :257
    return true;
}
template <int SMALL, bool STATS>
PTD_FI bool path_after_hit(const Ctx& c, bool hit, const Hit& h, Ray& r, uint32_t& seed, V3& radiance, V3& mask, int i,
                           int max_depth, SampleStats<STATS>& st, uint32_t visits) {
    PathRegs ps{r, seed, radiance, mask, {}};
    return path_after_hit<SMALL, STATS>(c, hit, h, ps, i, max_depth, st, visits);
}

// One iteration of the path loop, GenerateColors.cl:229-258: the scene query, then path_after_hit.
template <bool BVH, int SMALL, bool STATS>
PTD_FI bool path_segment(const Ctx& c, Ray& r, uint32_t& seed, V3& radiance, V3& mask, int i, int max_depth,
                         SampleStats<STATS>& st, RayCount& rc, QueryStats& qs) {
    Hit h;
    const uint32_t v0 = qs.visits;
    const bool hit = q_closest<BVH, SMALL, STATS>(c, r.o, r.d, h, qs);
    rc.closest++;
    return path_after_hit<SMALL, STATS>(c, hit, h, r, seed, radiance, mask, i, max_depth, st, qs.visits - v0);
}

// GenerateColors.cl:223-261 with BOUNCES -> max_depth
template <bool BVH, int SMALL, bool STATS>
PTD_FI V3 trace_rays(const Ctx& c, Ray r, uint32_t& seed, int max_depth, SampleStats<STATS>& st, RayCount& rc,
                     QueryStats& qs) {
    V3 radiance = mk(0.0f, 0.0f, 0.0f);  // :225
    V3 mask = mk(1.0f, 1.0f, 1.0f);      // :226
    for (int i = 0; i < max_depth; ++i)  // :229
        if (!path_segment<BVH, SMALL, STATS>(c, r, seed, radiance, mask, i, max_depth, st, rc, qs)) break;
    return mk(cl_max(radiance.x, 0.0f), cl_max(radiance.y, 0.0f), cl_max(radiance.z, 0.0f));  // :260
}

// BUILD-DEFINED C1
template <bool BVH, int SMALL, bool STATS>
PTD_FI V3 sample_primary(const Ctx& c, Ray r, SampleStats<STATS>& st, RayCount& rc, QueryStats& qs) {
    Hit h;
    const bool hit = q_closest<BVH, SMALL, STATS>(c, r.o, r.d, h, qs);
    rc.closest++;
    V3 p1, e1, e2; int idx = -1, quad = -1;
    if (hit) load_tri<SMALL>(c, h.pos, p1, e1, e2, idx, quad);
    st_primary(st, hit, h, quad, qs.visits);
    if constexpr (STATS) st.count = 1;
    if (!hit) return mk(0.45f, 0.45f, 0.45f);
    V3 albedo, emissive; float roughness; int type;
    load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);
    return albedo;
}

// BUILD-DEFINED C2
template <bool BVH, int SMALL, bool STATS>
PTD_FI V3 sample_ao(const Ctx& c, Ray r, uint32_t& seed, int ns, float max_dist, SampleStats<STATS>& st,
                    RayCount& rc, QueryStats& qs) {
    Hit h;
    const bool hit = q_closest<BVH, SMALL, STATS>(c, r.o, r.d, h, qs);
    rc.closest++;
    V3 p1, e1, e2; int idx = -1, quad = -1;
    if (hit) load_tri<SMALL>(c, h.pos, p1, e1, e2, idx, quad);
    st_primary(st, hit, h, quad, qs.visits);
    if (!hit) return mk(1.0f, 1.0f, 1.0f);
    V3 p, n;
    hit_point_normal(e1, e2, r.o, r.d, h, p, n);
    n = dot(n, r.d) < 0.0f ? n : mul(n, -1.0f);
    uint32_t open = 0;
    const Frame fr = make_frame(n);  // one tangent frame for all AO rays of the pixel
    for (int k = 0; k < ns; ++k) {
        const V3 wi = sample_hemisphere_cosine(n, fr, seed);
        const Ray s = get_ray(add(p, mul(wi, 0.01f)), wi);
        Hit b;
        const uint32_t v0 = qs.visits;
        const bool occ = q_any<BVH, SMALL, STATS>(c, s.o, s.d, max_dist, b, qs);
        rc.any++;
        st_secondary(st, occ ? b.idx : -1, qs.visits - v0);
        if (!occ) open++;
    }
    if constexpr (STATS) st.count = open;
    const float v = (float)open / (float)ns;
    return mk(v, v, v);
}

// BUILD-DEFINED C3
template <bool BVH, int SMALL, bool STATS>
PTD_FI V3 sample_direct(const Ctx& c, const RenderArgs& a, Ray r, uint32_t& seed, SampleStats<STATS>& st,
                        RayCount& rc, QueryStats& qs) {
    Hit h;
    const bool hit = q_closest<BVH, SMALL, STATS>(c, r.o, r.d, h, qs);
    rc.closest++;
    V3 p1, e1, e2; int idx = -1, quad = -1;
    if (hit) load_tri<SMALL>(c, h.pos, p1, e1, e2, idx, quad);
    st_primary(st, hit, h, quad, qs.visits);
    if (!hit) return mk(0.45f, 0.45f, 0.45f);
    V3 albedo, emissive; float roughness; int type;
    load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);
    V3 p, n;
    hit_point_normal(e1, e2, r.o, r.d, h, p, n);
    V3 col = mk(1.0f * emissive.x * 3.0f, 1.0f * emissive.y * 3.0f, 1.0f * emissive.z * 3.0f);
    n = dot(n, r.d) < 0.0f ? n : mul(n, -1.0f);
    const V3 wo = neg(r.d);
    const float xi1 = random_float(seed);
    const float xi2 = random_float(seed);
    const V3 lp = mk(a.light_p1[0], a.light_p1[1], a.light_p1[2]);
    const V3 ea = mk(a.light_ea[0], a.light_ea[1], a.light_ea[2]);
    const V3 eb = mk(a.light_eb[0], a.light_eb[1], a.light_eb[2]);
    const V3 P = add(add(lp, mul(ea, xi1)), mul(eb, xi2));
    const V3 L = sub(P, p);
    const float dist2 = dot(L, L);
    const float dist = sqrt_rn(dist2);
    const V3 wi = mul(L, rcp_rn(dist));  // == normalize(L): L * (1 / sqrt(dot(L, L)))
    const float area = a.light_area;
    const V3 nl = mk(a.light_n[0], a.light_n[1], a.light_n[2]);
    const float cos_s = dot(wi, n);
    const float cos_l = -dot(wi, nl);
    if (cos_s > 0.0f && cos_l > 0.0f) {
        const Ray s = get_ray(add(p, mul(wi, 0.01f)), wi);
        Hit b;
        const uint32_t v0 = qs.visits;
        const bool occ = q_any<BVH, SMALL, STATS>(c, s.o, s.d, dist - 0.02f, b, qs);
        rc.any++;
        st_secondary(st, occ ? b.idx : -1, qs.visits - v0);
        if (!occ) {
            if constexpr (STATS) st.count = 1;
            V3 lalb, lem; float lr; int lt;
            load_mat<SMALL>(c, a.light_quad, lalb, lr, lem, lt);
            V3 f;
            if (type == PTB_SPECULAR) {
                const V3 wh = normalize(add(wo, wi));
                const float D = distribution_ggx(dot(n, wh), roughness);
                const float k = D / (4.0f * dot(wi, n) * dot(wo, n));
                f = mk(k * albedo.x * 2.0f, k * albedo.y * 2.0f, k * albedo.z * 2.0f);
            } else {
                f = mul(albedo, PTD_INV_PI);
            }
            const float G = cos_s * cos_l / dist2;
            col = mk(col.x + f.x * (lem.x * 3.0f) * G * area, col.y + f.y * (lem.y * 3.0f) * G * area,
                     col.z + f.z * (lem.z * 3.0f) * G * area);
        }
    }
    return mk(cl_max(col.x, 0.0f), cl_max(col.y, 0.0f), cl_max(col.z, 0.0f));
}

// ---- megakernel: one thread per sample ---------------------------------------------------------

template <int MODE, bool BVH, int SMALL, bool STATS, class SRC = CameraRays>
__global__ void __launch_bounds__(128, ((MODE == PTB_MODE_AO || MODE == PTB_MODE_DIRECT) && BVH && SMALL) ? 8 : 0) k_mega(const SceneDev sc, const typename SRC::Args a) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<BVH, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (BVH && !SMALL && sc.lstack) c.lstack = lstack_mem;

    const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)a.frames_in_batch * a.n_local;
    RayCount rc{0u, 0u};
    QueryStats qs{0u, 0u};
    const bool valid = slot < total;
    if (valid) {
        int li, frame;
        uint32_t seed;
        Ray r;
        if constexpr (SRC::buffer) {
            li = (int)slot;
            frame = 0;
            load_sample_ray(a, slot, r, seed);
        } else {
            const int fi = (int)(slot / a.n_local);
            li = (int)(slot - (long long)fi * a.n_local);
            const int gid = gid_of_local(a.shard, li);
            frame = a.first_frame + fi;
            const int gi = gid % a.width, gj = gid / a.width;  // GenerateColors.cl:305-306
            seed = (uint32_t)gid + hash_uint32((uint32_t)frame);  // :308
            r = generate_ray(gi, gj, CamScale{a.cam_inv_w, a.cam_inv_h, a.cam_aspect}, seed);   // :310
        }
        SampleStats<STATS> st{};
        V3 col;
        if (MODE == PTB_MODE_PRIMARY) col = sample_primary<BVH, SMALL, STATS>(c, r, st, rc, qs);
        else if (MODE == PTB_MODE_AO) col = sample_ao<BVH, SMALL, STATS>(c, r, seed, a.ao_samples, a.ao_max_dist, st, rc, qs);
        else if (MODE == PTB_MODE_DIRECT) col = sample_direct<BVH, SMALL, STATS>(c, a, r, seed, st, rc, qs);
        else col = trace_rays<BVH, SMALL, STATS>(c, r, seed, a.max_depth, st, rc, qs);  // :312
        a.samples[slot] = make_float4(col.x, col.y, col.z, 1.0f);
        if constexpr (STATS) {
            if (a.stats && (SRC::buffer || frame == a.stats_frame)) {
                uint4* dst = reinterpret_cast<uint4*>(a.stats + li);
                dst[0] = make_uint4((uint32_t)st.tri, (uint32_t)st.quad, st.t_bits, st.visits_primary);
                dst[1] = make_uint4(st.visits_secondary, st.count, st.id_hash, qs.tests);
            }
        }
    }
    flush_counter(a.counters, CTR_CLOSEST, rc.closest);
    flush_counter(a.counters, CTR_ANY, rc.any);
    if (STATS) {
        flush_counter(a.counters, CTR_NODES, qs.visits);
        flush_counter(a.counters, CTR_TESTS, qs.tests);
    }
}

// ---- path megakernel with path regeneration ---------------------------------------------------------
// Paths end at different depths (miss through the open front, pdf <= 0, depth limit); with one sample per
// thread a warp idles its finished lanes until its longest path ends (Cornell, depth 8: 3.6 of 8 segments
// on average).  Here the grid is persistent and a lane whose path ended immediately draws the next sample
// slot from a global counter (one warp-aggregated atomicAdd per refill), so every warp iteration is one
// path segment for (nearly) 32 live lanes.  Per-sample arithmetic is unchanged -> identical results.
// COOP (FLAT scenes only): the triangle phase of the query is pooled over the warp (flat_mt_coop)
template <bool BVH, int SMALL, bool STATS, bool COOP = false, class SRC = CameraRays>
__global__ void __launch_bounds__(128, (COOP && !STATS) ? 9 : 0) k_mega_path_regen(const SceneDev sc, const typename SRC::Args a,
                                                         unsigned long long* work_counter) {
    static_assert(!COOP || (BVH && SMALL == PTD_FLAT), "the pooled triangle phase belongs to the FLAT query");
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<BVH, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (BVH && !SMALL && sc.lstack) c.lstack = lstack_mem;
    const long long total = (long long)a.frames_in_batch * a.n_local;
    const unsigned lane = threadIdx.x & 31u;
    RayCount rc{0u, 0u};
    QueryStats qs{0u, 0u};
    bool alive = false, done = false;
    long long slot = 0;
    int li = 0, frame = 0, depth = 0;
    uint32_t seed = 0, tests0 = 0;
    Ray r{mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f)};
    V3 radiance = mk(0.f, 0.f, 0.f), mask = mk(1.f, 1.f, 1.f);
    SampleStats<STATS> st{};
    for (;;) {
        const unsigned need = __ballot_sync(0xffffffffu, !alive && !done);
        // Regenerate when at least 6 lanes wait (or none is alive): camera-ray generation is ~250 instructions and ran at 9 of
        // 32 lanes when triggered by the first idle lane (C4 +2 %; 4: +1.2 %, 8: +2.0 %, 12: +0.7 %, 16: -1.8 %).  tune[0] = n
        // overrides the threshold (1 = as soon as one lane waits).  Scheduling only: per-sample arithmetic is unchanged.
        const unsigned live = __ballot_sync(0xffffffffu, alive);
        if (need && (live == 0u || __popc(need) >= (a.tune[0] > 0 ? a.tune[0] : 6))) {
            const int leader = __ffs(need) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned long long)__popc(need));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (!alive && !done) {
                slot = (long long)base + __popc(need & ((1u << lane) - 1u));
                if (slot >= total) {
                    done = true;
                } else {
                    if constexpr (SRC::buffer) {
                        li = (int)slot;
                        load_sample_ray(a, slot, r, seed);
                    } else {
                        const int fi = (int)(slot / a.n_local);
                        li = (int)(slot - (long long)fi * a.n_local);
                        const int gid = gid_of_local(a.shard, li);
                        frame = a.first_frame + fi;
                        seed = (uint32_t)gid + hash_uint32((uint32_t)frame);                    // GenerateColors.cl:308
                        r = generate_ray(gid % a.width, gid / a.width, CamScale{a.cam_inv_w, a.cam_inv_h, a.cam_aspect}, seed);  // :310
                    }
                    radiance = mk(0.f, 0.f, 0.f);
                    mask = mk(1.f, 1.f, 1.f);
                    depth = 0;
                    alive = true;
                    st = SampleStats<STATS>{};
                    tests0 = qs.tests;
                }
            }
        }
        if (!__any_sync(0xffffffffu, alive)) break;
        Hit ch;  // COOP (FLAT scenes): the query runs warp-cooperatively -- all lanes enter --, then the live lanes shade
        bool chit = false;
        uint32_t cvisits = 0;
        if constexpr (COOP) {
            unsigned long long tm = 0ull;
            const uint32_t v0 = qs.visits;
            if (alive) tm = flat_boxes<STATS>(c, r.o, r.d, 1e20f, qs);
            cvisits = qs.visits - v0;
            const unsigned long long key = flat_mt_coop<false>(c, c.s_coop, alive, r.o, r.d, 1e20f, tm, ch.u, ch.v);
            if (STATS) qs.tests += (uint32_t)__popcll(tm);
            chit = alive && key != ~0ull;
            ch.t = __uint_as_float((uint32_t)(key >> 32));
            ch.pos = (int)(key & 255u); ch.idx = chit ? (int)((key >> 8) & 0xffffffu) : -1;
        }
        if (alive) {
            bool more;
            if constexpr (COOP) {
                rc.closest++;
                more = path_after_hit<SMALL, STATS>(c, chit, ch, r, seed, radiance, mask, depth, a.max_depth, st, cvisits);
            } else {
                more = path_segment<BVH, SMALL, STATS>(c, r, seed, radiance, mask, depth, a.max_depth, st, rc, qs);
            }
            ++depth;
            if (!more || depth >= a.max_depth) {
                a.samples[slot] = make_float4(cl_max(radiance.x, 0.0f), cl_max(radiance.y, 0.0f), cl_max(radiance.z, 0.0f), 1.0f);  // :260
                if constexpr (STATS) {
                    if (a.stats && (SRC::buffer || frame == a.stats_frame)) {
                        uint4* dst = reinterpret_cast<uint4*>(a.stats + li);
                        dst[0] = make_uint4((uint32_t)st.tri, (uint32_t)st.quad, st.t_bits, st.visits_primary);
                        dst[1] = make_uint4(st.visits_secondary, st.count, st.id_hash, qs.tests - tests0);
                    }
                }
                alive = false;
            }
        }
    }
    flush_counter(a.counters, CTR_CLOSEST, rc.closest);
    if (STATS) {
        flush_counter(a.counters, CTR_NODES, qs.visits);
        flush_counter(a.counters, CTR_TESTS, qs.tests);
    }
}

// ---- path kernel as a per-lane state machine ("phase voting") ---------------------------------------------------------
// k_mega_path_regen keeps the classic while-while query inside one path segment: a warp leaves the node loop only when its
// slowest lane reached a leaf and leaves the segment only when its slowest query ended.  On a deep tree with incoherent rays
// the per-ray node count is heavy-tailed (2M-triangle scene: 23.7 on average, several times that for rays grazing a
// tessellated wall), so the node loop ran at 11 of 32 lanes (profiles/r02/ncu_k_mega_path_regen_c5_before_blocks.txt).
// Here every lane carries an explicit state and the WARP votes which phase runs next:
//     NODE   ONE node visit (tree forms) / the leaf-box sweep (FLAT)        } the inner "walk" loop: runs until thr_shade
//     LEAF   ONE triangle test, then the next triangle of the leaf or a pop  } lanes finished their query (or nobody walks)
//     SHADE  the part of the path loop after the query (path_after_hit)
//     REGEN  draw the next sample slot, generate the camera ray   (>= thr_regen lanes wait, or nothing else is left to do)
// so a phase runs for all lanes that need it, lanes of other states wait at most until their own phase collects its quorum,
// and a ray that walks 200 nodes no longer holds 31 finished lanes.  Per ray the order of node visits, triangle tests,
// culling and RNG draws is exactly bvh_query's / path_segment's -> results, visit and test counts are bit-identical.
// States are one-hot BYTES of one word, so that ONE warp reduction (REDUX.SUM) counts the lanes of all states at once.
enum : uint32_t { ST_DONE = 0u, ST_REGEN = 1u, ST_NODE = 1u << 8, ST_LEAF = 1u << 16, ST_SHADE = 1u << 24 };

// Visit of a (quantised) BINARY node from global memory with the stack in local memory (the 2M-triangle scene's form).  Same
// rule as node_step2 (DESIGN.md "Traversal order") with the common outcomes free of divergent paths: every lane fetches its node
// with ONE 256-bit load and, speculatively, its stack top together; descend / push / pop-of-a-live-entry are selects and one
// predicated store.  Only a pop that meets culled entries (entry distance > best_t) loops.  False = the query finished.
template <bool STATS>
PTD_FI bool node_step2_bf(const Ctx& c, const RayPre& rp, float best_t, int& cur, int& sp, QueryStats& qs) {
    uint4 a, b;
    ldg_nodeq(c.g_nodes, cur, a, b);
    const uint2 top = c.lstack[sp - 1];  // sp = 0 reads the spare slot below the stack (value unused): no clamp, the -1 folds into the address
    if (STATS) qs.visits++;
    float tn0, tn1;
    const bool h0 = qslab(a.x, a.y, a.z, rp, best_t, tn0);
    const bool h1 = qslab(a.w, b.x, b.y, rp, best_t, tn1);
    const int c0 = (int)b.z, c1 = (int)b.w;
    const bool second_first = tn1 < tn0;
    const bool both = h0 && h1;
    if (both) c.lstack[sp] = make_uint2((uint32_t)(second_first ? c0 : c1), __float_as_uint(second_first ? tn0 : tn1));
    if (h0 || h1) {
        cur = both ? (second_first ? c1 : c0) : (h0 ? c0 : c1);
        sp += both ? 1 : 0;
        return true;
    }
    if (sp == 0) return false;
    --sp;
    cur = (int)top.x;
    if (__uint_as_float(top.y) <= best_t) return true;
    while (sp > 0) {  // culled entries
        --sp;
        const uint2 e = c.lstack[sp];
        cur = (int)e.x;
        if (__uint_as_float(e.y) <= best_t) return true;
    }
    return false;
}

template <int SMALL, bool STATS, int MINB, int NSTEP = 1>
__global__ void __launch_bounds__(128, MINB) k_path_sm(const SceneDev sc, const RenderArgs a, unsigned long long* work_counter) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<true, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES + 1];  // [0] = spare slot below the stack (node_step2_bf reads the top speculatively)
    if (!SMALL && sc.lstack) c.lstack = lstack_mem + 1;
    const bool fast_nodes = SMALL == PTD_LARGE && sc.lstack && sc.smem_nodes == 0;  // warp-uniform: node_step2_bf applies
    const long long total = (long long)a.frames_in_batch * a.n_local;
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t thr_regen = a.tune[0] > 0 ? a.tune[0] : 6;
    const uint32_t thr_shade = a.tune[10] > 0 ? a.tune[10] : 16;
    const uint32_t thr_leaf = a.tune[11] > 0 ? a.tune[11] : 10;
    RayCount rc{0u, 0u};
    QueryStats qs{0u, 0u};
    uint32_t state = ST_REGEN;
    bool exhausted = false;  // warp-uniform: the work counter ran past the last sample slot
    long long slot = 0;
    int li = 0, frame = 0, depth = 0;
    uint32_t seed = 0, tests0 = 0, visits0 = 0;
    Ray r{mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f)};
    V3 radiance = mk(0.f, 0.f, 0.f), mask = mk(1.f, 1.f, 1.f);
    // query state
    RayPre rp{mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 0.f), {0u, 0u, 0u}};
    float best_t = 1e20f, best_u = 0.f, best_v = 0.f;
    int best_pos = -1, best_idx = -1, cur = 0, sp = 0;
    unsigned long long tm = 0ull;  // FLAT: triangles still to test
    SampleStats<STATS> st{};
    auto begin_query = [&]() {  // the ray in `r` starts its closest-hit query (bvh_query's / flat_query's preamble)
        visits0 = qs.visits;
        best_t = 1e20f; best_u = best_v = 0.f; best_pos = best_idx = -1;
        if constexpr (SMALL != PTD_FLAT) {
            rp = ray_pre<SMALL>(c, r.o, r.d);
            cur = 0; sp = 0;
        }
        state = ST_NODE;
    };
    for (;;) {
        // ---- walk: node visits and triangle tests until thr_shade lanes have finished their query, or nobody walks
        for (;;) {
            const uint32_t cnt = __reduce_add_sync(0xffffffffu, state);
            const uint32_t n_node = (cnt >> 8) & 255u, n_leaf = (cnt >> 16) & 255u, n_shade = cnt >> 24;
            if (n_leaf >= thr_leaf || (n_leaf && !n_node)) {
                if (state == ST_LEAF) {
                    int k;
                    if constexpr (SMALL == PTD_FLAT) {
                        k = __ffsll((long long)tm) - 1;
                        tm &= tm - 1ull;
                    } else {
                        k = (int)((uint32_t)(~cur) >> 3);
                    }
                    V3 p1, e1, e2; int idx, quad;
                    load_tri<SMALL>(c, k, p1, e1, e2, idx, quad);
                    float t, u, v;
                    if (STATS) qs.tests++;
                    if (mt_core(r.o, r.d, p1, e1, e2, t, u, v) && (t < best_t || (t == best_t && best_idx >= 0 && idx < best_idx))) {
                        best_t = t; best_u = u; best_v = v; best_pos = k; best_idx = idx;
                    }
                    if constexpr (SMALL == PTD_FLAT) {
                        if (!tm) state = ST_SHADE;
                    } else {
                        const uint32_t code = (uint32_t)(~cur);
                        if (code & 7u) cur = (int)~(((code >> 3) + 1u) << 3 | ((code & 7u) - 1u));  // the next triangle of this leaf
                        else if (stack_pop<false>(c, sp, cur, best_t)) state = cur >= 0 ? ST_NODE : ST_LEAF;
                        else state = ST_SHADE;
                    }
                }
                continue;
            }
            if (!n_node || n_shade >= thr_shade) break;
            if (state == ST_NODE) {
                if constexpr (SMALL == PTD_FLAT) {
                    tm = flat_boxes<STATS>(c, r.o, r.d, 1e20f, qs);
                    state = tm ? ST_LEAF : ST_SHADE;
                } else {
                    bool more;
                    if (SMALL == PTD_LARGE && fast_nodes) {
                        // NSTEP visits per vote (a lane that reaches a leaf or ends its query sits the rest out): the vote and its
                        // dispatch are a quarter of a single-visit iteration.  C5: 1 -> 3.73, 2 -> 3.95, 4 -> 4.08, 6 -> 4.11, 8 -> 3.96 Grays/s;
                        // re-voting adaptively (while 5/8..7/8 of the lanes are still at a node) measured 3.86..3.99.
                        more = node_step2_bf<STATS>(c, rp, best_t, cur, sp, qs);
#pragma unroll
                        for (int rep = 1; rep < NSTEP; ++rep)
                            if (more && cur >= 0) more = node_step2_bf<STATS>(c, rp, best_t, cur, sp, qs);
                    }
                    else more = node_step<false, SMALL, STATS>(c, rp, best_t, cur, sp, qs);
                    state = !more ? ST_SHADE : cur >= 0 ? ST_NODE : ST_LEAF;
                }
            }
        }
        // ---- shade every lane whose query finished
        if (state == ST_SHADE) {
            Hit h;
            const bool hit = best_idx >= 0;
            h.t = best_t; h.u = best_u; h.v = best_v; h.pos = best_pos; h.idx = best_idx;
            rc.closest++;
            const bool more = path_after_hit<SMALL, STATS>(c, hit, h, r, seed, radiance, mask, depth, a.max_depth, st, qs.visits - visits0);
            ++depth;
            if (!more || depth >= a.max_depth) {
                a.samples[slot] = make_float4(cl_max(radiance.x, 0.0f), cl_max(radiance.y, 0.0f), cl_max(radiance.z, 0.0f), 1.0f);  // :260
                if constexpr (STATS) {
                    if (a.stats && frame == a.stats_frame) {
                        uint4* dst = reinterpret_cast<uint4*>(a.stats + li);
                        dst[0] = make_uint4((uint32_t)st.tri, (uint32_t)st.quad, st.t_bits, st.visits_primary);
                        dst[1] = make_uint4(st.visits_secondary, st.count, st.id_hash, qs.tests - tests0);
                    }
                }
                state = exhausted ? ST_DONE : ST_REGEN;
            } else {
                begin_query();
            }
        }
        // ---- new samples for the lanes whose path ended: when thr_regen of them wait, or when nothing else is left to do
        const unsigned m_regen = __ballot_sync(0xffffffffu, state == ST_REGEN);
        const unsigned m_walk = __ballot_sync(0xffffffffu, (state & (ST_NODE | ST_LEAF)) != 0u);
        const uint32_t n_regen = __popc(m_regen);
        if (n_regen && (n_regen >= thr_regen || !m_walk)) {  // (lanes are never in REGEN once `exhausted` is set)
            const int leader = __ffs(m_regen) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned long long)n_regen);
            base = __shfl_sync(0xffffffffu, base, leader);
            if ((long long)base + (long long)n_regen >= total) exhausted = true;
            if (state == ST_REGEN) {
                slot = (long long)base + __popc(m_regen & ((1u << lane) - 1u));
                if (slot >= total) {
                    state = ST_DONE;
                } else {
                    const int fi = (int)(slot / a.n_local);
                    li = (int)(slot - (long long)fi * a.n_local);
                    const int gid = gid_of_local(a.shard, li);
                    frame = a.first_frame + fi;
                    seed = (uint32_t)gid + hash_uint32((uint32_t)frame);                    // GenerateColors.cl:308
                    r = generate_ray(gid % a.width, gid / a.width, CamScale{a.cam_inv_w, a.cam_inv_h, a.cam_aspect}, seed);  // :310
                    radiance = mk(0.f, 0.f, 0.f);
                    mask = mk(1.f, 1.f, 1.f);
                    depth = 0;
                    st = SampleStats<STATS>{};
                    tests0 = qs.tests;
                    begin_query();
                }
            }
        } else if (!m_walk) {
            break;  // nobody walks, nobody waits for a sample, every query was shaded: all lanes are DONE
        }
    }
    flush_counter(a.counters, CTR_CLOSEST, rc.closest);
    if (STATS) {
        flush_counter(a.counters, CTR_NODES, qs.visits);
        flush_counter(a.counters, CTR_TESTS, qs.tests);
    }
}

// ---- k_path_sm with the path state parked in shared memory ------------------------------------------------------------
// The walk loop of k_path_sm needs the box-test constants, best_t, the current reference and the stack height; everything
// else a lane carries (ray, hit record, radiance, mask, seed, slot, depth: 19 words) is only touched by the triangle test,
// the shade phase and the regeneration.  Here those words live in a per-thread shared-memory column (conflict-free: word f of
// thread t at f * 512 + t * 4), loaded where a phase needs them, so the walk loop fits a lower register cap and more CTAs are
// resident per SM (the kernel hides dependent-load latency with resident warps: 8 -> 7 CTAs cost 7.5 %).  Large scenes with the
// local-memory stack and no staged prefix only; per-sample arithmetic and order unchanged.  Measured on C5 (same kernel body,
// 6 visits per vote): registers only, 8 CTAs 4.36 Grays/s; parked, 8 / 9 / 10 / 11 CTAs (64 / 56 / 48 / 40 registers): 4.43 / 4.58 /
// 4.61 / 4.62 with the old quorums, 4.69 at 10 CTAs with the re-tuned ones.
// A node visit or a shade step runs only for the lanes in that state, but registers belong to threads: whatever one lane keeps in
// registers across a phase, every lane pays for.  So the box-test constants (RayPre, 9 words) live in the column too: written once
// per query by begin_query and loaded by the node phase at each vote; and the shading step (path_after_hit over PathCol) loads each
// field where it uses it and stores it back as soon as it is final.  At the 40-register cap of 12 CTAs per SM nothing spills
// (it spilled 128 B per thread when RayPre and the loaded path state were held across the shade phase).
enum { PK_OX = 0, PK_OY, PK_OZ, PK_DX, PK_DY, PK_DZ, PK_U, PK_V, PK_POS, PK_IDX, PK_RX, PK_RY, PK_RZ, PK_MX, PK_MY, PK_MZ, PK_SEED, PK_SLOT, PK_DEPTH,
       PK_AX, PK_AY, PK_AZ, PK_BX, PK_BY, PK_BZ, PK_SN0, PK_SN1, PK_SN2, PK_FIELDS };
static inline size_t path_sm2_smem_bytes(int block) { return 16 + (size_t)PK_FIELDS * block * 4; }
constexpr uint32_t PK_STRIDE = 128u * 4u;  // the launcher runs k_path_sm2 with 128-thread CTAs only: field offsets are immediates

// path_after_hit's path state in a lane's shared-memory column (pk: the address of its word 0).  Each field is loaded where the
// shading step uses it and stored as soon as it is final, so that no field stays in a register across the step.
struct PathCol {
    uint32_t pk;
    Ray r;  // the last ray set_ray stored, for the query that follows
    PTD_FI float ldf(int f) const { return __uint_as_float(lds32(pk + (uint32_t)f * PK_STRIDE)); }
    PTD_FI void stf(int f, float v) const { sts32(pk + (uint32_t)f * PK_STRIDE, __float_as_uint(v)); }
    PTD_FI V3 o() const { return mk(ldf(PK_OX), ldf(PK_OY), ldf(PK_OZ)); }
    PTD_FI V3 d() const { return mk(ldf(PK_DX), ldf(PK_DY), ldf(PK_DZ)); }
    PTD_FI uint32_t rng() const { return lds32(pk + PK_SEED * PK_STRIDE); }
    PTD_FI V3 rad() const { return mk(ldf(PK_RX), ldf(PK_RY), ldf(PK_RZ)); }
    PTD_FI V3 msk() const { return mk(ldf(PK_MX), ldf(PK_MY), ldf(PK_MZ)); }
    PTD_FI V3 hit_point() const { return o(); }  // the hit point replaces the origin, which is dead once it is known
    PTD_FI void set_rng(uint32_t v) { sts32(pk + PK_SEED * PK_STRIDE, v); }
    PTD_FI void set_rad(V3 v) { stf(PK_RX, v.x); stf(PK_RY, v.y); stf(PK_RZ, v.z); }
    PTD_FI void set_msk(V3 v) { stf(PK_MX, v.x); stf(PK_MY, v.y); stf(PK_MZ, v.z); }
    PTD_FI void set_hit_point(V3 v) { stf(PK_OX, v.x); stf(PK_OY, v.y); stf(PK_OZ, v.z); }
    PTD_FI void set_ray(const Ray& v) {
        r = v;
        stf(PK_OX, v.o.x); stf(PK_OY, v.o.y); stf(PK_OZ, v.o.z); stf(PK_DX, v.d.x); stf(PK_DY, v.d.y); stf(PK_DZ, v.d.z);
    }
};

// The body of k_path_sm2 for either ray source (k_path_sm2: the camera; k_path_sm2_rays: a caller's ptb_sample_ray buffer).
template <bool STATS, int NSTEP, class SRC>
PTD_FI void path_sm2(const SceneDev& sc, const typename SRC::Args& a, unsigned long long* work_counter) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<true, PTD_LARGE>(sc, smem);  // stages nothing (smem_nodes == 0): only the Ctx
    uint2 lstack_mem[PTD_LSTACK_ENTRIES + 1];
    c.lstack = lstack_mem + 1;
    uint32_t pk = smem_u32(smem) + 16u + threadIdx.x * 4u;
    asm volatile("" : "+r"(pk));  // opaque: kept in a register instead of being re-derived (S2R + shared-window base + LEA, 7 instructions) at every vote
#define PKL(f) lds32(pk + (uint32_t)(f) * PK_STRIDE)
#define PKLF(f) __uint_as_float(lds32(pk + (uint32_t)(f) * PK_STRIDE))
#define PKS(f, v) sts32(pk + (uint32_t)(f) * PK_STRIDE, (uint32_t)(v))
#define PKSF(f, v) sts32(pk + (uint32_t)(f) * PK_STRIDE, __float_as_uint(v))
    const uint32_t total = (uint32_t)((long long)a.frames_in_batch * a.n_local);  // the launcher guarantees < 2^31 slots
    const unsigned lane = threadIdx.x & 31u;
    // quorums, resolved by the launcher (defaults re-tuned for 10 resident CTAs: shade 16 / 20 / 24 -> 4.61 / 4.66 / 4.51,
    // regen 4 / 6 / 8 -> 4.69 / 4.66 / 4.59 Grays/s): plain kernel parameters, no select in the loop
    const uint32_t thr_regen = (uint32_t)a.tune[0], thr_shade = (uint32_t)a.tune[10], thr_leaf = (uint32_t)a.tune[11];
    RayCount rc{0u, 0u};
    QueryStats qs{0u, 0u};
    uint32_t state = ST_REGEN;
    bool exhausted = false;
    int li = 0, frame = 0;  // STATS only
    uint32_t tests0 = 0, visits0 = 0;
    float best_t = 1e20f;
    int cur = 0, sp = 0;
    SampleStats<STATS> st{};
    auto begin_query = [&](const Ray& r) {
        visits0 = qs.visits;
        best_t = 1e20f;
        PKS(PK_IDX, -1);
        const RayPre q = ray_pre<PTD_LARGE>(c, r.o, r.d);
        PKSF(PK_AX, q.a.x); PKSF(PK_AY, q.a.y); PKSF(PK_AZ, q.a.z); PKSF(PK_BX, q.b.x); PKSF(PK_BY, q.b.y); PKSF(PK_BZ, q.b.z);
        PKS(PK_SN0, q.sn[0]); PKS(PK_SN1, q.sn[1]); PKS(PK_SN2, q.sn[2]);
        cur = 0; sp = 0;
        state = ST_NODE;
    };
    for (;;) {
        for (;;) {
            const uint32_t cnt = __reduce_add_sync(0xffffffffu, state);
            const uint32_t n_node = (cnt >> 8) & 255u, n_leaf = (cnt >> 16) & 255u, n_shade = cnt >> 24;
            if (n_leaf >= thr_leaf || (n_leaf && !n_node)) {
                if (state == ST_LEAF) {
                    const int k = (int)((uint32_t)(~cur) >> 3);
                    V3 p1, e1, e2; int idx, quad;
                    load_tri<PTD_LARGE>(c, k, p1, e1, e2, idx, quad);
                    const V3 o = mk(PKLF(PK_OX), PKLF(PK_OY), PKLF(PK_OZ)), d = mk(PKLF(PK_DX), PKLF(PK_DY), PKLF(PK_DZ));
                    float t, u, v;
                    if (STATS) qs.tests++;
                    if (mt_core(o, d, p1, e1, e2, t, u, v)) {
                        bool take = t < best_t;
                        if (t == best_t) { const int bi = (int)PKL(PK_IDX); take = bi >= 0 && idx < bi; }
                        if (take) {
                            best_t = t;
                            PKSF(PK_U, u); PKSF(PK_V, v); PKS(PK_POS, k); PKS(PK_IDX, idx);
                        }
                    }
                    const uint32_t code = (uint32_t)(~cur);
                    if (code & 7u) cur = (int)~(((code >> 3) + 1u) << 3 | ((code & 7u) - 1u));
                    else if (stack_pop<false>(c, sp, cur, best_t)) state = cur >= 0 ? ST_NODE : ST_LEAF;
                    else state = ST_SHADE;
                }
                continue;
            }
            if (!n_node || n_shade >= thr_shade) break;
            if (state == ST_NODE) {
                const RayPre rp{mk(PKLF(PK_AX), PKLF(PK_AY), PKLF(PK_AZ)), mk(PKLF(PK_BX), PKLF(PK_BY), PKLF(PK_BZ)), {PKL(PK_SN0), PKL(PK_SN1), PKL(PK_SN2)}};
                bool more = node_step2_bf<STATS>(c, rp, best_t, cur, sp, qs);
#pragma unroll
                for (int rep = 1; rep < NSTEP; ++rep)
                    if (more && cur >= 0) more = node_step2_bf<STATS>(c, rp, best_t, cur, sp, qs);
                state = !more ? ST_SHADE : cur >= 0 ? ST_NODE : ST_LEAF;
            }
        }
        if (state == ST_SHADE) {
            Hit h;
            h.idx = (int)PKL(PK_IDX);
            const bool hit = h.idx >= 0;
            h.t = best_t; h.u = PKLF(PK_U); h.v = PKLF(PK_V); h.pos = (int)PKL(PK_POS);
            const int depth = (int)PKL(PK_DEPTH);
            rc.closest++;
            PathCol ps{pk, {}};
            const bool more = path_after_hit<PTD_LARGE, STATS>(c, hit, h, ps, depth, a.max_depth, st, qs.visits - visits0);
            if (!more || depth + 1 >= a.max_depth) {
                const V3 radiance = ps.rad();
                a.samples[PKL(PK_SLOT)] = make_float4(cl_max(radiance.x, 0.0f), cl_max(radiance.y, 0.0f), cl_max(radiance.z, 0.0f), 1.0f);  // :260
                if constexpr (STATS) {
                    if (a.stats && (SRC::buffer || frame == a.stats_frame)) {
                        uint4* dst = reinterpret_cast<uint4*>(a.stats + li);
                        dst[0] = make_uint4((uint32_t)st.tri, (uint32_t)st.quad, st.t_bits, st.visits_primary);
                        dst[1] = make_uint4(st.visits_secondary, st.count, st.id_hash, qs.tests - tests0);
                    }
                }
                state = exhausted ? ST_DONE : ST_REGEN;
            } else {
                PKS(PK_DEPTH, depth + 1);
                begin_query(ps.r);
            }
        }
        const unsigned m_regen = __ballot_sync(0xffffffffu, state == ST_REGEN);
        const unsigned m_walk = __ballot_sync(0xffffffffu, (state & (ST_NODE | ST_LEAF)) != 0u);
        const uint32_t n_regen = __popc(m_regen);
        if (n_regen && (n_regen >= thr_regen || !m_walk)) {
            const int leader = __ffs(m_regen) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned long long)n_regen);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + n_regen >= (unsigned long long)total) exhausted = true;
            if (state == ST_REGEN) {
                const unsigned long long slot = base + __popc(m_regen & ((1u << lane) - 1u));
                if (slot >= (unsigned long long)total) {
                    state = ST_DONE;
                } else {
                    uint32_t seed;
                    Ray r;
                    if constexpr (SRC::buffer) {
                        li = (int)slot;
                        load_sample_ray(a, (long long)slot, r, seed);
                    } else {
                        const int fi = (int)(slot / (unsigned)a.n_local);
                        const int l = (int)(slot - (unsigned long long)fi * (unsigned)a.n_local);
                        const int gid = gid_of_local(a.shard, l);
                        li = l; frame = a.first_frame + fi;
                        seed = (uint32_t)gid + hash_uint32((uint32_t)(a.first_frame + fi));  // GenerateColors.cl:308
                        r = generate_ray(gid % a.width, gid / a.width, CamScale{a.cam_inv_w, a.cam_inv_h, a.cam_aspect}, seed);  // :310
                    }
                    PKSF(PK_OX, r.o.x); PKSF(PK_OY, r.o.y); PKSF(PK_OZ, r.o.z); PKSF(PK_DX, r.d.x); PKSF(PK_DY, r.d.y); PKSF(PK_DZ, r.d.z);
                    PKSF(PK_RX, 0.0f); PKSF(PK_RY, 0.0f); PKSF(PK_RZ, 0.0f); PKSF(PK_MX, 1.0f); PKSF(PK_MY, 1.0f); PKSF(PK_MZ, 1.0f);
                    PKS(PK_SEED, seed); PKS(PK_SLOT, (uint32_t)slot); PKS(PK_DEPTH, 0);
                    st = SampleStats<STATS>{};
                    tests0 = qs.tests;
                    begin_query(r);
                }
            }
        } else if (!m_walk) {
            break;
        }
    }
#undef PKL
#undef PKLF
#undef PKS
#undef PKSF
    flush_counter(a.counters, CTR_CLOSEST, rc.closest);
    if (STATS) {
        flush_counter(a.counters, CTR_NODES, qs.visits);
        flush_counter(a.counters, CTR_TESTS, qs.tests);
    }
}

template <bool STATS, int MINB, int NSTEP>
__global__ void __launch_bounds__(128, MINB) k_path_sm2(const SceneDev sc, const RenderArgs a, unsigned long long* work_counter) {
    path_sm2<STATS, NSTEP, CameraRays>(sc, a, work_counter);
}
// ptb_scene_shade: the same kernel on the sample rays of a caller's buffer, under a name of its own (k_path_sm2 keeps its symbol)
template <bool STATS, int MINB, int NSTEP>
__global__ void __launch_bounds__(128, MINB) k_path_sm2_rays(const SceneDev sc, const ShadeArgs a, unsigned long long* work_counter) {
    path_sm2<STATS, NSTEP, SampleRays>(sc, a, work_counter);
}

// ---- ordered accumulation of a batch: GenerateColors.cl:290-321 --------------------------------

PTD_FI V3 gamma_correct(V3 v) {  // :290-294
    const float g = 1.0f / 2.2f;
    return mk(det_pow(v.x, g), det_pow(v.y, g), det_pow(v.z, g));
}
PTD_FI V3 read_from_gamma(V3 v) {  // :296-300
    return mk(det_pow(v.x, 2.2f), det_pow(v.y, 2.2f), det_pow(v.z, 2.2f));
}

struct ResolveArgs {
    const float4* samples;
    int n_local, frames_in_batch, first_frame;
    int accum;
    int first_batch, last_batch;
    int total_frames;
    float4* sum;    // linear running sum (xyz)
    float4* frame;  // output / gamma-space state
    // gather mode (ptb_render_gather): `frame` and `peers[]` are FULL images indexed by the global pixel id; the resolved
    // pixel is stored into this rank's image and into every peer's (their memory is mapped over NVLink)
    int gather, n_peers;
    Shard shard;
    float4* peers[PTB_MAX_PEERS];
};

PTD_FI void resolve_store(const ResolveArgs& a, size_t at, float4 v) {
    a.frame[at] = v;
    for (int k = 0; k < a.n_peers; ++k) a.peers[k][at] = v;  // 16-byte remote stores, coalesced per 64-pixel block
}

__global__ void __launch_bounds__(256) k_resolve(const ResolveArgs a) {
    const int li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= a.n_local) return;
    const size_t at = a.gather ? (size_t)gid_of_local(a.shard, li) : (size_t)li;
    if (a.accum == PTB_ACCUM_REFERENCE) {
        float4 cur = a.frame[at];
        V3 state = xyz(cur);
        float w = cur.w;
        for (int fi = 0; fi < a.frames_in_batch; ++fi) {
            const V3 col = xyz(a.samples[(size_t)fi * a.n_local + li]);
            const int f = a.first_frame + fi;
            if (f == 0) {  // :314-317
                state = gamma_correct(col);
            } else {       // :318-321
                const V3 prev = read_from_gamma(state);
                const float zm1 = (float)(f - 1), z = (float)f;
                state = gamma_correct(mk((prev.x * zm1 + col.x) / z, (prev.y * zm1 + col.y) / z, (prev.z * zm1 + col.z) / z));
            }
            w = 1.0f;
        }
        resolve_store(a, at, make_float4(state.x, state.y, state.z, w));
    } else {
        V3 s = a.first_batch ? mk(0.0f, 0.0f, 0.0f) : xyz(a.sum[li]);
        for (int fi = 0; fi < a.frames_in_batch; ++fi) {
            const V3 col = xyz(a.samples[(size_t)fi * a.n_local + li]);
            s = mk(s.x + col.x, s.y + col.y, s.z + col.z);
        }
        if (a.last_batch) {
            const float nf = (float)a.total_frames;
            resolve_store(a, at, make_float4(s.x / nf, s.y / nf, s.z / nf, 1.0f));
        } else {
            a.sum[li] = make_float4(s.x, s.y, s.z, 0.0f);
        }
    }
}

// ---- output transform on the device: RaytraceTest.cpp:78-83 f2c applied to sqrtf(v) (:283) ----------------------
// Same arithmetic as ptb_to_rgb8 (scene.cpp): IEEE sqrt, one multiply, truncation, clamp; out-of-int-range values
// follow the x86 conversion (INT_MIN -> 0), NaN -> 0.  Four pixels per thread = three 32-bit stores.
PTD_FI uint32_t f2c_sqrt(float v) {
    const float a = sqrtf(v) * 255.0f;
    if (!(a == a)) return 0u;
    if (a >= 2147483648.0f || a < -2147483648.0f) return 0u;
    const int b = (int)a;
    return (uint32_t)(b > 255 ? 255 : (b < 0 ? 0 : b));
}
__global__ void __launch_bounds__(256) k_to_rgb8(const float4* frame, int n, uint8_t* rgb) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;  // group of four pixels
    const int i0 = q * 4;
    if (i0 >= n) return;
    if (i0 + 4 <= n) {
        uint32_t b[12];
        for (int k = 0; k < 4; ++k) {
            const float4 v = frame[i0 + k];
            b[3 * k] = f2c_sqrt(v.x); b[3 * k + 1] = f2c_sqrt(v.y); b[3 * k + 2] = f2c_sqrt(v.z);
        }
        uint32_t* dst = reinterpret_cast<uint32_t*>(rgb + (size_t)i0 * 3);  // 12-byte groups from a 16-byte aligned base
        dst[0] = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24);
        dst[1] = b[4] | (b[5] << 8) | (b[6] << 16) | (b[7] << 24);
        dst[2] = b[8] | (b[9] << 8) | (b[10] << 16) | (b[11] << 24);
    } else {
        for (int i = i0; i < n; ++i) {
            const float4 v = frame[i];
            rgb[(size_t)i * 3] = (uint8_t)f2c_sqrt(v.x); rgb[(size_t)i * 3 + 1] = (uint8_t)f2c_sqrt(v.y); rgb[(size_t)i * 3 + 2] = (uint8_t)f2c_sqrt(v.z);
        }
    }
}

// ---- scene queries on caller-supplied rays (tests) -----------------------------------------------

struct TraceArgs {
    int n_rays;
    const float* o;
    const float* d;
    const float* tmax;
    int* out_tri;
    float* out_t;
    float* out_u;
    float* out_v;
    uint32_t* out_visits;
    uint32_t* out_tests;
};

template <bool BVH, bool ANY, int SMALL>
__global__ void __launch_bounds__(128) k_trace(const SceneDev sc, const TraceArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<BVH, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (BVH && !SMALL && sc.lstack) c.lstack = lstack_mem;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_rays) return;
    const V3 o = mk(a.o[3 * i], a.o[3 * i + 1], a.o[3 * i + 2]);
    const V3 d = mk(a.d[3 * i], a.d[3 * i + 1], a.d[3 * i + 2]);
    Hit h;
    h.t = h.u = h.v = 0.0f; h.pos = h.idx = -1;
    QueryStats qs{0u, 0u};
    bool hit;
    if (ANY) hit = q_any<BVH, SMALL, true>(c, o, d, a.tmax[i], h, qs);
    else hit = q_closest<BVH, SMALL, true>(c, o, d, h, qs);
    a.out_tri[i] = hit ? h.idx : -1;
    a.out_t[i] = hit ? h.t : 0.0f;
    a.out_u[i] = hit ? h.u : 0.0f;
    a.out_v[i] = hit ? h.v : 0.0f;
    a.out_visits[i] = qs.visits;
    a.out_tests[i] = qs.tests;
}

// ---- unit kernels for the numerics contract -------------------------------------------------------

__global__ void k_test_sincos(const float* x, int n, float* s, float* c) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) det_sincos(x[i], s[i], c[i]);
}
__global__ void k_test_pow(const float* x, int n, float y, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = det_pow(x[i], y);
}
// out[0..n) = rcp_rn(x), out[n..2n) = sqrt_rn(x), out[2n..3n) = safe_rcp3(x,x,x).x, out[3n..6n) = normalize(x, 0.5x, 2x)
__global__ void k_test_ieee(const float* x, int n, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = x[i];
    out[i] = rcp_rn(v);
    out[(size_t)n + i] = sqrt_rn(v);
    out[2 * (size_t)n + i] = safe_rcp3(mk(v, v, v)).x;
    const V3 u = normalize(mk(v, 0.5f * v, 2.0f * v));
    out[3 * (size_t)n + i] = u.x; out[4 * (size_t)n + i] = u.y; out[5 * (size_t)n + i] = u.z;
}
__global__ void k_test_rng(uint32_t gid, uint32_t frame, int n, uint32_t* states, float* values) {
    if (blockIdx.x || threadIdx.x) return;
    uint32_t seed = gid + hash_uint32(frame);
    for (int i = 0; i < n; ++i) {
        values[i] = random_float(seed);
        states[i] = seed;
    }
}
__global__ void k_test_camera(int width, int height, int frame, int n, const int* gids, float* o, float* d,
                              uint32_t* seeds) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int gid = gids[i];
    uint32_t seed = (uint32_t)gid + hash_uint32((uint32_t)frame);
    const Ray r = generate_ray(gid % width, gid / width, width, height, seed);
    o[3 * i] = r.o.x; o[3 * i + 1] = r.o.y; o[3 * i + 2] = r.o.z;
    d[3 * i] = r.d.x; d[3 * i + 1] = r.d.y; d[3 * i + 2] = r.d.z;
    seeds[i] = seed;
}

}  // namespace ptd
