// pt_wavefront.cuh -- wavefront integrator: the same per-sample arithmetic as the
// megakernel (pt_kernels.cuh), split into stages that each run SIMT-dense over a
// queue of live rays:
//
//   wf_generate      camera ray + RNG seed per path slot            (GenerateColors.cl:305-310)
//   wf_extend        closest-hit scene query per queued ray          (:137-154 / BVH)
//   wf_shade_*       material, emission, BSDF sample, next ray       (:233-257)
//                    -> surviving paths are appended to the next queue with
//                       warp-aggregated atomics (one atomicAdd per warp)
//   wf_shadow_*      any-hit query per shadow / AO ray
//   wf_finish_*      per-slot combination of shadow results
//
// Queue records are SoA float4 streams (coalesced 128-bit accesses):
//   q_o = (origin.xyz, slot)  q_d = (dir.xyz, seed)  q_m = (mask.xyz, has_radiance)
//   hit = (t, u, v, triangle position | -1)
// A path slot = (frame-in-batch, local pixel); each slot's radiance lands in
// samples[slot], so k_resolve accumulates in frame order exactly as for the
// megakernel and both integrators are bit-identical.
#pragma once

#include "host_internal.h"
#include "pt_kernels.cuh"

namespace ptd {

struct WfBuffers {
    float4* q_o[2];
    float4* q_d[2];
    float4* q_m[2];
    float4* hit;
    float4* radiance;        // running radiance of slots that met an emitter and went on
    float4* slot_p;          // AO: hit point per slot; DIRECT: base colour per slot
    float4* sq_w;            // AO: (wi.xyz, tmax | <0 hole); DIRECT: (o.xyz, tmax | <0 hole)
    float4* sq_d;            // DIRECT: (d.xyz, -)
    float4* sq_c;            // DIRECT: (contribution.xyz, -)
    int* sq_res;             // per shadow ray: blocker triangle index, -1 = unoccluded, -2 = hole
    uint32_t* sq_visits;     // STATS
    uint32_t* sq_tests;      // STATS
    ptb_pixel_stats* slot_stats;  // STATS: per slot
    unsigned int* counts;    // queue lengths: counts[d] = rays entering depth d
    unsigned int* work;      // persistent kernels: next ray index, one counter per launch
};

PTD_FI bool finite3(V3 v) {
    return fabsf(v.x) <= 3.402823466e38f && fabsf(v.y) <= 3.402823466e38f && fabsf(v.z) <= 3.402823466e38f;
}

// ---- generate ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wf_generate(const RenderArgs a, const WfBuffers w, const int stats) {
    const long long total = (long long)a.frames_in_batch * a.n_local;
    const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot == 0) w.counts[0] = (unsigned int)total;
    if (slot >= total) return;
    const int fi = (int)(slot / a.n_local);
    const int li = (int)(slot - (long long)fi * a.n_local);
    const int gid = gid_of_local(a.shard, li);
    const int frame = a.first_frame + fi;
    uint32_t seed = (uint32_t)gid + hash_uint32((uint32_t)frame);          // GenerateColors.cl:308
    const Ray r = generate_ray(gid % a.width, gid / a.width, CamScale{a.cam_inv_w, a.cam_inv_h, a.cam_aspect}, seed);  // :310
    w.q_o[0][slot] = make_float4(r.o.x, r.o.y, r.o.z, __int_as_float((int)slot));
    w.q_d[0][slot] = make_float4(r.d.x, r.d.y, r.d.z, __uint_as_float(seed));
    w.q_m[0][slot] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
    if (stats) {
        uint4* s = reinterpret_cast<uint4*>(w.slot_stats + slot);
        s[0] = make_uint4(0xffffffffu, 0xffffffffu, 0u, 0u);
        s[1] = make_uint4(0u, 0u, 0u, 0u);
    }
}

// ---- extend --------------------------------------------------------------------------------------
template <bool BVH, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_extend(const SceneDev sc, const WfBuffers w, const int depth, const int qi,
                                                 unsigned long long* counters) {
    const unsigned int n = w.counts[depth];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<BVH, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (BVH && !SMALL && sc.lstack) c.lstack = lstack_mem;
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t nrays = 0;
    QueryStats qs{0u, 0u};
    if (i < n) {
        const float4 qo = w.q_o[qi][i], qd = w.q_d[qi][i];
        Hit h;
        const bool hit = q_closest<BVH, SMALL, STATS>(c, xyz(qo), xyz(qd), h, qs);
        nrays = 1;
        w.hit[i] = make_float4(h.t, h.u, h.v, __int_as_float(hit ? h.pos : -1));
        if constexpr (STATS) {
            ptb_pixel_stats* s = w.slot_stats + __float_as_int(qo.w);
            if (depth == 0) {
                int quad = -1;
                if (hit) {
                    V3 p1, e1, e2; int idx;
                    load_tri<SMALL>(c, h.pos, p1, e1, e2, idx, quad);
                }
                s->tri = hit ? h.idx : -1;
                s->quad = quad;
                s->t_bits = hit ? __float_as_uint(h.t) : 0u;
                s->visits_primary = qs.visits;
            } else {
                s->visits_secondary += qs.visits;
                s->id_hash = s->id_hash * 31u + (uint32_t)((hit ? h.idx : -1) + 2);
            }
            s->tri_tests += qs.tests;
        }
    }
    flush_counter(counters, CTR_CLOSEST, nrays);
    if (STATS) {
        flush_counter(counters, CTR_NODES, qs.visits);
        flush_counter(counters, CTR_TESTS, qs.tests);
    }
}

// ---- persistent while-while traversal with dynamic ray fetch ---------------------------------------
// One warp keeps 32 traversal states.  A lane whose ray ended becomes idle; when a warp vote finds at
// least `refill_thr` idle lanes (or none traversing) the idle lanes draw fresh ray indices from a global
// work counter with ONE warp-aggregated atomicAdd and re-arm.  Between refills the classic while-while
// runs: internal nodes until no lane has one, then the leaves.  Per-ray traversal (order, visit counts,
// results) is exactly bvh_query's; only which lanes run together changes.
//   IO::load(i, o, d, tmax) -> false for a hole;  IO::store(i, hit, h, qs) publishes one ray's result.
template <bool ANY, int SMALL, bool STATS, class IO>
PTD_FI void trace_persistent(const Ctx& c, IO& io, const unsigned int n_rays, unsigned int* work_counter,
                             const int refill_thr, uint32_t& n_traced, QueryStats& total) {
    const unsigned lane = threadIdx.x & 31u;
    bool active = false;
    bool exhausted = false;  // warp-uniform
    unsigned int idx = 0;
    V3 o = mk(0.f, 0.f, 0.f), d = o;
    RayPre rp{o, o, {0u, 0u, 0u}};
    float best_t = 0.f, best_u = 0.f, best_v = 0.f;
    int best_pos = -1, best_idx = -1, cur = 0, sp = 0;
    QueryStats qs{0u, 0u};
    for (;;) {
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (idle != 0u && !exhausted && (idle == 0xffffffffu || __popc(idle) >= refill_thr)) {
            const int leader = __ffs(idle) - 1;
            unsigned int base = 0;
            if ((int)lane == leader) base = atomicAdd(work_counter, (unsigned int)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (!active) {
                idx = base + (unsigned int)__popc(idle & ((1u << lane) - 1u));
                float tmax;
                if (idx < n_rays && io.load(idx, o, d, tmax)) {
                    rp = ray_pre<SMALL>(c, o, d);
                    best_t = tmax; best_u = best_v = 0.f; best_pos = best_idx = -1;
                    cur = 0; sp = 0;
                    qs.visits = qs.tests = 0u;
                    active = true;
                    ++n_traced;
                }
            }
            if (base + (unsigned int)__popc(idle) >= n_rays) exhausted = true;
        }
        unsigned act = __ballot_sync(0xffffffffu, active);
        if (act == 0u) {
            if (exhausted) break;
            continue;
        }
        for (;;) {
            bool fin = false, blocked = false;
            Hit h;
            while (active && !fin && cur >= 0)
                if (!node_step<ANY, SMALL, STATS>(c, rp, best_t, cur, sp, qs)) fin = true;
            if (active && !fin) {  // leaf
                const uint32_t code = (uint32_t)(~cur);
                const int first = (int)(code >> 3), count = (int)(code & 7u) + 1;
                for (int k = first; k < first + count; ++k) {
                    V3 p1, e1, e2; int tidx, quad;
                    load_tri<SMALL>(c, k, p1, e1, e2, tidx, quad);
                    float t, u, v;
                    if (STATS) qs.tests++;
                    if (!mt_core(o, d, p1, e1, e2, t, u, v)) continue;
                    if (ANY) {
                        if (t < best_t) { best_t = t; best_u = u; best_v = v; best_pos = k; best_idx = tidx; blocked = true; break; }
                    } else if (t < best_t || (t == best_t && best_idx >= 0 && tidx < best_idx)) {
                        best_t = t; best_u = u; best_v = v; best_pos = k; best_idx = tidx;
                    }
                }
                if (blocked || !stack_pop<ANY>(c, sp, cur, best_t)) fin = true;
            }
            if (active && fin) {
                const bool hit = ANY ? blocked : best_idx >= 0;
                h.t = best_t; h.u = best_u; h.v = best_v; h.pos = best_pos; h.idx = hit ? best_idx : -1;
                io.store(idx, hit, h, qs);
                if (STATS) { total.visits += qs.visits; total.tests += qs.tests; }
                active = false;
            }
            act = __ballot_sync(0xffffffffu, active);
            if (act == 0u) break;
            if (!exhausted && 32 - __popc(act) >= refill_thr) break;
        }
    }
}

// The same persistent traversal as a per-lane state machine (see k_path_sm): the warp votes whether the next step is a
// refill (>= refill_thr lanes idle), ONE triangle test for the lanes at a leaf (>= thr_leaf of them, or nobody at a node) or
// ONE node visit for the others, so a lane on a long walk never waits for the leaves of its neighbours and a fresh ray's
// long first descent does not stall lanes that are between two leaves.  Per ray the sequence of node visits, triangle tests
// and culls is bvh_query's: results and counts are identical.  Used for scenes traversed from L2/HBM.
template <bool ANY, int SMALL, bool STATS, class IO>
PTD_FI void trace_persistent_sm(const Ctx& c, IO& io, const unsigned int n_rays, unsigned int* work_counter,
                                const uint32_t refill_thr, const uint32_t thr_leaf, const bool fast_nodes, uint32_t& n_traced,
                                QueryStats& total) {
    const unsigned lane = threadIdx.x & 31u;
    uint32_t state = ST_REGEN;  // ST_REGEN = idle: the lane wants a ray
    bool exhausted = false;     // warp-uniform
    unsigned int idx = 0;
    V3 o = mk(0.f, 0.f, 0.f), d = o;
    RayPre rp{o, o, {0u, 0u, 0u}};
    float best_t = 0.f, best_u = 0.f, best_v = 0.f;
    int best_pos = -1, best_idx = -1, cur = 0, sp = 0;
    bool blocked = false;
    QueryStats qs{0u, 0u};
    auto finish = [&]() {
        Hit h;
        const bool hit = ANY ? blocked : best_idx >= 0;
        h.t = best_t; h.u = best_u; h.v = best_v; h.pos = best_pos; h.idx = hit ? best_idx : -1;
        io.store(idx, hit, h, qs);
        if (STATS) { total.visits += qs.visits; total.tests += qs.tests; }
        state = ST_REGEN;
    };
    for (;;) {
        const uint32_t cnt = __reduce_add_sync(0xffffffffu, state);
        const uint32_t n_idle = cnt & 255u, n_node = (cnt >> 8) & 255u, n_leaf = (cnt >> 16) & 255u;
        const bool walking = (n_node | n_leaf) != 0u;
        if (!exhausted && n_idle && (n_idle >= refill_thr || !walking)) {
            const unsigned idle = __ballot_sync(0xffffffffu, state == ST_REGEN);
            const int leader = __ffs(idle) - 1;
            unsigned int base = 0;
            if ((int)lane == leader) base = atomicAdd(work_counter, n_idle);
            base = __shfl_sync(0xffffffffu, base, leader);
            if (state == ST_REGEN) {
                idx = base + (unsigned int)__popc(idle & ((1u << lane) - 1u));
                float tmax;
                if (idx < n_rays && io.load(idx, o, d, tmax)) {
                    rp = ray_pre<SMALL>(c, o, d);
                    best_t = tmax; best_u = best_v = 0.f; best_pos = best_idx = -1;
                    cur = 0; sp = 0; blocked = false;
                    qs.visits = qs.tests = 0u;
                    state = ST_NODE;
                    ++n_traced;
                }
            }
            if (base + n_idle >= n_rays) exhausted = true;
            continue;
        }
        if (n_leaf >= thr_leaf || (n_leaf && !n_node)) {
            if (state == ST_LEAF) {
                const uint32_t code = (uint32_t)(~cur);
                const int k = (int)(code >> 3);
                V3 p1, e1, e2; int tidx, quad;
                load_tri<SMALL>(c, k, p1, e1, e2, tidx, quad);
                float t, u, v;
                if (STATS) qs.tests++;
                if (mt_core(o, d, p1, e1, e2, t, u, v)) {
                    if (ANY) {
                        if (t < best_t) { best_t = t; best_u = u; best_v = v; best_pos = k; best_idx = tidx; blocked = true; }
                    } else if (t < best_t || (t == best_t && best_idx >= 0 && tidx < best_idx)) {
                        best_t = t; best_u = u; best_v = v; best_pos = k; best_idx = tidx;
                    }
                }
                if (ANY && blocked) finish();
                else if (code & 7u) cur = (int)~(((code >> 3) + 1u) << 3 | ((code & 7u) - 1u));  // the next triangle of this leaf
                else if (stack_pop<ANY>(c, sp, cur, best_t)) state = cur >= 0 ? ST_NODE : ST_LEAF;
                else finish();
            }
            continue;
        }
        if (!n_node) break;  // nobody walks and the idle lanes cannot be refilled
        if (state == ST_NODE) {
            bool more;
            if (!ANY && SMALL == PTD_LARGE && fast_nodes) more = node_step2_bf<STATS>(c, rp, best_t, cur, sp, qs);
            else more = node_step<ANY, SMALL, STATS>(c, rp, best_t, cur, sp, qs);
            if (!more) finish();
            else state = cur >= 0 ? ST_NODE : ST_LEAF;
        }
    }
}

struct ExtendIO {
    const float4* qo;
    const float4* qd;
    float4* hit;
    ptb_pixel_stats* slot_stats;
    int depth;
    int slot;  // of the ray this lane holds
    PTD_FI bool load(unsigned int i, V3& o, V3& d, float& tmax) {
        const float4 a = qo[i], b = qd[i];
        o = xyz(a); d = xyz(b);
        slot = __float_as_int(a.w);
        tmax = 1e20f;
        return true;
    }
};

template <int SMALL, bool STATS>
struct ExtendStore : ExtendIO {
    const Ctx* c;
    PTD_FI void store(unsigned int i, bool hit_any, const Hit& h, const QueryStats& qs) {
        hit[i] = make_float4(h.t, h.u, h.v, __int_as_float(hit_any ? h.pos : -1));
        if constexpr (STATS) {
            ptb_pixel_stats* s = slot_stats + slot;
            if (depth == 0) {
                int quad = -1;
                if (hit_any) {
                    V3 p1, e1, e2; int idx;
                    load_tri<SMALL>(*c, h.pos, p1, e1, e2, idx, quad);
                }
                s->tri = hit_any ? h.idx : -1;
                s->quad = quad;
                s->t_bits = hit_any ? __float_as_uint(h.t) : 0u;
                s->visits_primary = qs.visits;
            } else {
                s->visits_secondary += qs.visits;
                s->id_hash = s->id_hash * 31u + (uint32_t)((hit_any ? h.idx : -1) + 2);
            }
            s->tri_tests += qs.tests;
        }
    }
};

template <int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_extend_p(const SceneDev sc, const WfBuffers w, const int depth, const int qi,
                                                   unsigned long long* counters, const int refill_thr, const int sm_thr_leaf) {
    const unsigned int n = w.counts[depth];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<true, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES + 1];  // [0] = spare slot below the stack (node_step2_bf reads the top speculatively)
    if (!SMALL && sc.lstack) c.lstack = lstack_mem + 1;
    ExtendStore<SMALL, STATS> io;
    io.qo = w.q_o[qi]; io.qd = w.q_d[qi]; io.hit = w.hit; io.slot_stats = w.slot_stats; io.depth = depth; io.slot = 0;
    io.c = &c;
    uint32_t nrays = 0;
    QueryStats total{0u, 0u};
    // sm_thr_leaf > 0 (tune[13] = 1): the state-machine form for scenes traversed from L2/HBM; default: while-while
    if (SMALL == PTD_LARGE && sm_thr_leaf > 0)
        trace_persistent_sm<false, SMALL, STATS>(c, io, n, w.work + depth, (uint32_t)refill_thr, (uint32_t)sm_thr_leaf,
                                                 sc.lstack && sc.smem_nodes == 0, nrays, total);
    else
        trace_persistent<false, SMALL, STATS>(c, io, n, w.work + depth, refill_thr, nrays, total);
    flush_counter(counters, CTR_CLOSEST, nrays);
    if (STATS) {
        flush_counter(counters, CTR_NODES, total.visits);
        flush_counter(counters, CTR_TESTS, total.tests);
    }
}

template <int MODE, bool STATS>
struct ShadowIO {
    const RenderArgs* a;
    const WfBuffers* w;
    long long P;
    PTD_FI bool load(unsigned int i, V3& o, V3& d, float& tmax) {
        const float4 rw = w->sq_w[i];
        if (!(rw.w >= 0.0f || rw.w != rw.w)) {  // hole
            if (MODE == PTB_MODE_AO) w->sq_res[i] = -2;
            return false;
        }
        if (MODE == PTB_MODE_AO) {
            const V3 p = xyz(w->slot_p[(long long)i % P]);
            const V3 wi = xyz(rw);
            const Ray s = get_ray(add(p, mul(wi, 0.01f)), wi);
            o = s.o; d = s.d;
        } else {
            o = xyz(rw);
            d = xyz(w->sq_d[i]);
        }
        tmax = rw.w;
        return true;
    }
    PTD_FI void store(unsigned int i, bool occ, const Hit& h, const QueryStats& qs) {
        const int res = occ ? h.idx : -1;
        if (MODE == PTB_MODE_AO) {
            w->sq_res[i] = res;
            if constexpr (STATS) { w->sq_visits[i] = qs.visits; w->sq_tests[i] = qs.tests; }
        } else {
            V3 col = xyz(w->slot_p[i]);
            if (!occ) {
                const V3 cc = xyz(w->sq_c[i]);
                col = mk(col.x + cc.x, col.y + cc.y, col.z + cc.z);
            }
            a->samples[i] = make_float4(cl_max(col.x, 0.0f), cl_max(col.y, 0.0f), cl_max(col.z, 0.0f), 1.0f);
            if constexpr (STATS) {
                ptb_pixel_stats* s = w->slot_stats + i;
                s->visits_secondary += qs.visits;
                s->id_hash = s->id_hash * 31u + (uint32_t)(res + 2);
                s->tri_tests += qs.tests;
                if (!occ) s->count = 1;
            }
        }
    }
};

template <int MODE, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_shadow_p(const SceneDev sc, const RenderArgs a, const WfBuffers w,
                                                   const unsigned int n_rays, unsigned int* work,
                                                   unsigned long long* counters, const int refill_thr) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<true, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (!SMALL && sc.lstack) c.lstack = lstack_mem;
    ShadowIO<MODE, STATS> io;
    io.a = &a; io.w = &w; io.P = (long long)a.frames_in_batch * a.n_local;
    uint32_t nrays = 0;
    QueryStats total{0u, 0u};
    trace_persistent<true, SMALL, STATS>(c, io, n_rays, work, refill_thr, nrays, total);
    flush_counter(counters, CTR_ANY, nrays);
    if (STATS) {
        flush_counter(counters, CTR_NODES, total.visits);
        flush_counter(counters, CTR_TESTS, total.tests);
    }
}

// ---- scene queries on caller-owned ray buffers (ptb_scene_intersect) ------------------------------------
// One ptb_ray = (o.xyz, tmax)(d.xyz, -) read with ONE 256-bit load; one ptb_hit = (t, u, v, caller index | -1) written with ONE
// 128-bit store (t = u = v = 0 on a miss, as ptb_trace and the oracle report it); stats: (nodes fetched, triangle tests) per ray.
template <bool STATS>
struct RayBufIO {
    const float4* rays;  // 2 x float4 per ray
    float4* hits;
    uint2* stats;
    PTD_FI bool load(unsigned int i, V3& o, V3& d, float& tmax) {
        float4 a, b;
        ldg256(rays + 2 * (size_t)i, a, b);
        o = xyz(a); tmax = a.w; d = xyz(b);
        return true;
    }
    PTD_FI void store(unsigned int i, bool hit, const Hit& h, const QueryStats& qs) {
        hits[i] = hit ? make_float4(h.t, h.u, h.v, __int_as_float(h.idx)) : make_float4(0.0f, 0.0f, 0.0f, __int_as_float(-1));
        if constexpr (STATS) stats[i] = make_uint2(qs.visits, qs.tests);
    }
};

// Tree forms: the persistent while-while traversal of the wavefront stages (dynamic ray fetch, refill at 8 idle lanes); on the
// 2M-triangle scene it beat the state-machine form and one thread per ray on camera and any-hit rays and was within 1 % on
// incoherent closest-hit rays (DESIGN.md section 5).
// FLAT scenes have no node loop to keep busy: one thread per ray over flat_query, as the wavefront does for them.
template <bool ANY, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) k_intersect(const SceneDev sc, const float4* rays, float4* hits, uint2* stats,
                                                   const unsigned int n_rays, unsigned int* work, unsigned long long* counters) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<true, SMALL>(sc, smem);
    RayBufIO<STATS> io{rays, hits, stats};
    uint32_t nrays = 0;
    QueryStats total{0u, 0u};
    if constexpr (SMALL == PTD_FLAT) {
        const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n_rays) {
            V3 o, d;
            float tmax;
            io.load(i, o, d, tmax);
            Hit h;
            const bool hit = flat_query<ANY, STATS>(c, o, d, tmax, h, total);
            io.store(i, hit, h, total);
            nrays = 1;
        }
    } else {
        uint2 lstack_mem[PTD_LSTACK_ENTRIES];
        if (!SMALL && sc.lstack) c.lstack = lstack_mem;
        trace_persistent<ANY, SMALL, STATS>(c, io, n_rays, work, 8, nrays, total);
    }
    flush_counter(counters, ANY ? CTR_ANY : CTR_CLOSEST, nrays);
    if (STATS) {
        flush_counter(counters, CTR_NODES, total.visits);
        flush_counter(counters, CTR_TESTS, total.tests);
    }
}

// ---- shade: full path (GenerateColors.cl:233-257) ---------------------------------------------------
template <bool BVH, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_shade_path(const SceneDev sc, const RenderArgs a, const WfBuffers w,
                                                     const int depth, const int qi) {
    const unsigned int n = w.counts[depth];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(16) unsigned char smem[];
    const Ctx c = stage_scene<false, SMALL, BVH>(sc, smem);  // triangles (in the order extend searched) + materials
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool alive = false;
    float4 no = make_float4(0, 0, 0, 0), nd = no, nm = no;
    if (i < n) {
        const float4 qo = w.q_o[qi][i], qd = w.q_d[qi][i], qm = w.q_m[qi][i];
        const float4 hr = w.hit[i];
        const int slot = __float_as_int(qo.w);
        uint32_t seed = __float_as_uint(qd.w);
        const V3 o = xyz(qo), d = xyz(qd);
        V3 mask = xyz(qm);
        bool has_rad = qm.w != 0.0f;
        const int pos = __float_as_int(hr.w);
        if constexpr (STATS) w.slot_stats[slot].count++;
        V3 add_rad;
        bool terminate;
        if (pos < 0) {  // :233-237
            add_rad = mk(mask.x * 0.45f, mask.y * 0.45f, mask.z * 0.45f);
            terminate = true;
        } else {
            V3 p1, e1, e2; int idx, quad;
            load_tri<SMALL>(c, pos, p1, e1, e2, idx, quad);
            Hit h; h.t = hr.x; h.u = hr.y; h.v = hr.z; h.pos = pos; h.idx = idx;
            V3 p, nrm;
            hit_point_normal(e1, e2, o, d, h, p, nrm);
            V3 albedo, emissive; float roughness; int type;
            load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);                 // :239
            add_rad = mk(mask.x * emissive.x * 3.0f, mask.y * emissive.y * 3.0f, mask.z * emissive.z * 3.0f);  // :241
            terminate = depth + 1 >= a.max_depth;  // the last segment's BSDF sample cannot reach the radiance
            if (!terminate) {
                nrm = dot(nrm, d) < 0.0f ? nrm : mul(nrm, -1.0f);                       // :243
                V3 wi = mk(0.0f, 0.0f, 0.0f);
                const V3 wo = neg(d);                                                    // :246
                float pdf = 0.0f;
                const V3 color = brdf(wo, wi, pdf, nrm, albedo, roughness, type, seed);  // :249
                if (pdf <= 0.0f) {                                                       // :251
                    terminate = true;
                } else {
                    const float dw = dot(wi, nrm);
                    mask = mk(mask.x * (color.x * dw / pdf), mask.y * (color.y * dw / pdf), mask.z * (color.z * dw / pdf));
                    const Ray r = get_ray(add(p, mul(wi, 0.01f)), wi);                   // :257
                    no = make_float4(r.o.x, r.o.y, r.o.z, qo.w);
                    nd = make_float4(r.d.x, r.d.y, r.d.z, __uint_as_float(seed));
                    alive = true;
                }
            }
            // radiance + (+0) is the identity unless the mask is non-finite (0 * inf = NaN)
            const bool adds = emissive.x != 0.0f || emissive.y != 0.0f || emissive.z != 0.0f || !finite3(xyz(qm));
            if (!terminate && adds) {
                V3 rad = has_rad ? xyz(w.radiance[slot]) : mk(0.0f, 0.0f, 0.0f);
                rad = mk(rad.x + add_rad.x, rad.y + add_rad.y, rad.z + add_rad.z);
                w.radiance[slot] = make_float4(rad.x, rad.y, rad.z, 0.0f);
                has_rad = true;
            }
        }
        if (terminate) {
            V3 rad = has_rad ? xyz(w.radiance[slot]) : mk(0.0f, 0.0f, 0.0f);
            rad = mk(rad.x + add_rad.x, rad.y + add_rad.y, rad.z + add_rad.z);
            a.samples[slot] = make_float4(cl_max(rad.x, 0.0f), cl_max(rad.y, 0.0f), cl_max(rad.z, 0.0f), 1.0f);  // :260
        }
        nm = make_float4(mask.x, mask.y, mask.z, has_rad ? 1.0f : 0.0f);
    }
    // append survivors to the next queue: ballot per warp, ONE atomicAdd per CTA (a single hot counter
    // serialises in L2: at 4K, one atomic per warp was 260 k same-address atomics per launch)
    __shared__ unsigned int s_cnt[32];
    __shared__ unsigned int s_base;
    const unsigned int ballot = __ballot_sync(0xffffffffu, alive);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = (blockDim.x + 31) >> 5;
    if (lane == 0) s_cnt[warp] = (unsigned int)__popc(ballot);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int total = 0;
        for (int k = 0; k < n_warps; ++k) { const unsigned int v = s_cnt[k]; s_cnt[k] = total; total += v; }
        s_base = total ? atomicAdd(&w.counts[depth + 1], total) : 0u;
    }
    __syncthreads();
    if (alive) {
        const unsigned int dst = s_base + s_cnt[warp] + (unsigned int)__popc(ballot & ((1u << lane) - 1u));
        w.q_o[qi ^ 1][dst] = no;
        w.q_d[qi ^ 1][dst] = nd;
        w.q_m[qi ^ 1][dst] = nm;
    }
}

// ---- shade: primary / AO / direct -------------------------------------------------------------------
template <int MODE, bool BVH, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_shade_first(const SceneDev sc, const RenderArgs a, const WfBuffers w) {
    const unsigned int n = w.counts[0];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(16) unsigned char smem[];
    const Ctx c = stage_scene<false, SMALL, BVH>(sc, smem);
    const unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 qo = w.q_o[0][i], qd = w.q_d[0][i];
    const float4 hr = w.hit[i];
    const int slot = __float_as_int(qo.w);
    const long long P = (long long)a.frames_in_batch * a.n_local;
    uint32_t seed = __float_as_uint(qd.w);
    const V3 o = xyz(qo), d = xyz(qd);
    const int pos = __float_as_int(hr.w);
    if (MODE == PTB_MODE_PRIMARY) {
        if constexpr (STATS) w.slot_stats[slot].count = 1;
        if (pos < 0) { a.samples[slot] = make_float4(0.45f, 0.45f, 0.45f, 1.0f); return; }
        V3 p1, e1, e2; int idx, quad;
        load_tri<SMALL>(c, pos, p1, e1, e2, idx, quad);
        V3 albedo, emissive; float roughness; int type;
        load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);
        a.samples[slot] = make_float4(albedo.x, albedo.y, albedo.z, 1.0f);
        return;
    }
    if (MODE == PTB_MODE_AO) {
        const int ns = a.ao_samples;
        if (pos < 0) {
            a.samples[slot] = make_float4(1.0f, 1.0f, 1.0f, 1.0f);  // final
            for (int k = 0; k < ns; ++k) w.sq_w[(size_t)k * P + slot] = make_float4(0.f, 0.f, 0.f, -1.0f);
            return;
        }
        V3 p1, e1, e2; int idx, quad;
        load_tri<SMALL>(c, pos, p1, e1, e2, idx, quad);
        Hit h; h.t = hr.x; h.u = hr.y; h.v = hr.z; h.pos = pos; h.idx = idx;
        V3 p, nrm;
        hit_point_normal(e1, e2, o, d, h, p, nrm);
        nrm = dot(nrm, d) < 0.0f ? nrm : mul(nrm, -1.0f);
        a.samples[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // pending (w = 0)
        w.slot_p[slot] = make_float4(p.x, p.y, p.z, 0.0f);
        const Frame fr = make_frame(nrm);
        for (int k = 0; k < ns; ++k) {
            const V3 wi = sample_hemisphere_cosine(nrm, fr, seed);
            w.sq_w[(size_t)k * P + slot] = make_float4(wi.x, wi.y, wi.z, a.ao_max_dist);
        }
        return;
    }
    // DIRECT
    {
        w.sq_w[slot] = make_float4(0.f, 0.f, 0.f, -1.0f);
        if (pos < 0) { a.samples[slot] = make_float4(0.45f, 0.45f, 0.45f, 1.0f); return; }
        V3 p1, e1, e2; int idx, quad;
        load_tri<SMALL>(c, pos, p1, e1, e2, idx, quad);
        Hit h; h.t = hr.x; h.u = hr.y; h.v = hr.z; h.pos = pos; h.idx = idx;
        V3 albedo, emissive; float roughness; int type;
        load_mat<SMALL>(c, quad, albedo, roughness, emissive, type);
        V3 p, nrm;
        hit_point_normal(e1, e2, o, d, h, p, nrm);
        const V3 col = mk(1.0f * emissive.x * 3.0f, 1.0f * emissive.y * 3.0f, 1.0f * emissive.z * 3.0f);
        nrm = dot(nrm, d) < 0.0f ? nrm : mul(nrm, -1.0f);
        const V3 wo = neg(d);
        const float xi1 = random_float(seed);
        const float xi2 = random_float(seed);
        const V3 lp = mk(a.light_p1[0], a.light_p1[1], a.light_p1[2]);
        const V3 ea = mk(a.light_ea[0], a.light_ea[1], a.light_ea[2]);
        const V3 eb = mk(a.light_eb[0], a.light_eb[1], a.light_eb[2]);
        const V3 Pl = add(add(lp, mul(ea, xi1)), mul(eb, xi2));
        const V3 L = sub(Pl, p);
        const float dist2 = dot(L, L);
        const float dist = sqrt_rn(dist2);
        const V3 wi = mul(L, rcp_rn(dist));  // == normalize(L)
        const float area = a.light_area;
        const V3 nl = mk(a.light_n[0], a.light_n[1], a.light_n[2]);
        const float cos_s = dot(wi, nrm);
        const float cos_l = -dot(wi, nl);
        if (cos_s > 0.0f && cos_l > 0.0f) {
            const Ray s = get_ray(add(p, mul(wi, 0.01f)), wi);
            V3 lalb, lem; float lr; int lt;
            load_mat<SMALL>(c, a.light_quad, lalb, lr, lem, lt);
            V3 f;
            if (type == PTB_SPECULAR) {
                const V3 wh = normalize(add(wo, wi));
                const float D = distribution_ggx(dot(nrm, wh), roughness);
                const float k = D / (4.0f * dot(wi, nrm) * dot(wo, nrm));
                f = mk(k * albedo.x * 2.0f, k * albedo.y * 2.0f, k * albedo.z * 2.0f);
            } else {
                f = mul(albedo, PTD_INV_PI);
            }
            const float G = cos_s * cos_l / dist2;
            w.sq_w[slot] = make_float4(s.o.x, s.o.y, s.o.z, dist - 0.02f);
            w.sq_d[slot] = make_float4(s.d.x, s.d.y, s.d.z, 0.0f);
            w.sq_c[slot] = make_float4(f.x * (lem.x * 3.0f) * G * area, f.y * (lem.y * 3.0f) * G * area,
                                       f.z * (lem.z * 3.0f) * G * area, 0.0f);
            w.slot_p[slot] = make_float4(col.x, col.y, col.z, 0.0f);
        } else {
            a.samples[slot] = make_float4(cl_max(col.x, 0.0f), cl_max(col.y, 0.0f), cl_max(col.z, 0.0f), 1.0f);
        }
    }
}

// ---- shadow / AO any-hit stage -----------------------------------------------------------------------
template <int MODE, bool BVH, int SMALL, bool STATS>
__global__ void __launch_bounds__(128) wf_shadow(const SceneDev sc, const RenderArgs a, const WfBuffers w,
                                                 const long long n_rays, unsigned long long* counters) {
    extern __shared__ __align__(16) unsigned char smem[];
    Ctx c = stage_scene<BVH, SMALL>(sc, smem);
    uint2 lstack_mem[PTD_LSTACK_ENTRIES];
    if (BVH && !SMALL && sc.lstack) c.lstack = lstack_mem;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long P = (long long)a.frames_in_batch * a.n_local;
    uint32_t nrays = 0;
    QueryStats qs{0u, 0u};
    if (i < n_rays) {
        const float4 rw = w.sq_w[i];
        int res = -2;
        if (rw.w >= 0.0f || rw.w != rw.w) {  // holes carry tmax = -1
            V3 o, d;
            if (MODE == PTB_MODE_AO) {
                const long long slot = i % P;
                const V3 p = xyz(w.slot_p[slot]);
                const V3 wi = xyz(rw);
                const Ray s = get_ray(add(p, mul(wi, 0.01f)), wi);
                o = s.o; d = s.d;
            } else {
                o = xyz(rw);
                d = xyz(w.sq_d[i]);
            }
            Hit b;
            const bool occ = q_any<BVH, SMALL, STATS>(c, o, d, rw.w, b, qs);
            nrays = 1;
            res = occ ? b.idx : -1;
            if (MODE == PTB_MODE_DIRECT) {
                V3 col = xyz(w.slot_p[i]);
                if (!occ) {
                    const V3 cc = xyz(w.sq_c[i]);
                    col = mk(col.x + cc.x, col.y + cc.y, col.z + cc.z);
                }
                a.samples[i] = make_float4(cl_max(col.x, 0.0f), cl_max(col.y, 0.0f), cl_max(col.z, 0.0f), 1.0f);
                if constexpr (STATS) {
                    ptb_pixel_stats* s = w.slot_stats + i;
                    s->visits_secondary += qs.visits;
                    s->id_hash = s->id_hash * 31u + (uint32_t)(res + 2);
                    s->tri_tests += qs.tests;
                    if (!occ) s->count = 1;
                }
            }
        }
        if (MODE == PTB_MODE_AO) {
            w.sq_res[i] = res;
            if constexpr (STATS) { w.sq_visits[i] = qs.visits; w.sq_tests[i] = qs.tests; }
        }
    }
    flush_counter(counters, CTR_ANY, nrays);
    if (STATS) {
        flush_counter(counters, CTR_NODES, qs.visits);
        flush_counter(counters, CTR_TESTS, qs.tests);
    }
}

template <bool STATS>
__global__ void __launch_bounds__(256) wf_finish_ao(const RenderArgs a, const WfBuffers w) {
    const long long P = (long long)a.frames_in_batch * a.n_local;
    const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= P) return;
    if (a.samples[slot].w != 0.0f) return;  // primary miss: already final
    const int ns = a.ao_samples;
    uint32_t open = 0;
    for (int k = 0; k < ns; ++k) {
        const int res = w.sq_res[(size_t)k * P + slot];
        if (res == -1) open++;
        if constexpr (STATS) {
            ptb_pixel_stats* s = w.slot_stats + slot;
            s->visits_secondary += w.sq_visits[(size_t)k * P + slot];
            s->tri_tests += w.sq_tests[(size_t)k * P + slot];
            s->id_hash = s->id_hash * 31u + (uint32_t)(res + 2);
        }
    }
    if constexpr (STATS) w.slot_stats[slot].count = open;
    const float v = (float)open / (float)ns;
    a.samples[slot] = make_float4(v, v, v, 1.0f);
}

// copy the statistics of the slots that belong to stats_frame
__global__ void __launch_bounds__(256) wf_export_stats(const RenderArgs a, const WfBuffers w) {
    const int li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= a.n_local) return;
    const int fi = a.stats_frame - a.first_frame;
    if (fi < 0 || fi >= a.frames_in_batch) return;
    const uint4* s = reinterpret_cast<const uint4*>(w.slot_stats + (size_t)fi * a.n_local + li);
    uint4* d = reinterpret_cast<uint4*>(a.stats + li);
    d[0] = s[0];
    d[1] = s[1];
}

// ---- host orchestration ------------------------------------------------------------------------------

#define WF_TRY(expr)                                                                         \
    do {                                                                                     \
        cudaError_t e__ = (expr);                                                            \
        if (e__ != cudaSuccess) return ptb::fail(PTB_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

template <class K>
static int wf_smem(K kernel, size_t smem) {
    if (smem > 48 * 1024) WF_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
}

template <bool BVH, int SMALL, bool STATS>
static int wf_run(cudaStream_t st, int mode, const SceneDev& sc, const RenderArgs& a, const WfBuffers& w,
                  unsigned long long* counters, uint64_t* launches, int sm_count) {
    const long long P = (long long)a.frames_in_batch * a.n_local;
    const int block = 128;
    const unsigned grid = (unsigned)((P + block - 1) / block);
    // tune[6]=1: one thread per ray (no dynamic fetch).  FLAT scenes have no node loop to keep busy: one thread per ray.
    const bool persist = BVH && SMALL != PTD_FLAT && a.tune[6] == 0;
    const int refill_thr = a.tune[7] > 0 ? a.tune[7] : 8;  // idle lanes that trigger a refill
    // tune[13] = 1: the state-machine form of the extend stage for large scenes (lanes at a leaf that trigger a triangle step: tune[11], default 10);
    // default: while-while with dynamic fetch, which measures 3-7 % faster inside the wavefront integrator (C5, 16 frames per batch: 3.45 vs 3.21 Grays/s)
    const int sm_thr_leaf = a.tune[13] == 1 ? (a.tune[11] > 0 ? a.tune[11] : 10) : 0;
    auto pgrid = [&](auto kernel, size_t smem, long long n_items) -> unsigned {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
        long long g = (long long)per_sm * sm_count;
        const long long need = (n_items + block - 1) / block;
        return (unsigned)(g < need ? g : need);
    };
    const size_t smem_q = scene_smem_bytes(sc, BVH, SMALL, block);
    const size_t smem_s = scene_smem_bytes(sc, false, SMALL, block);
    int rc;
    wf_generate<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a, w, STATS ? 1 : 0);
    WF_TRY(cudaGetLastError());
    *launches += 1;
    auto ext = wf_extend<BVH, SMALL, STATS>;
    if ((rc = wf_smem(ext, smem_q))) return rc;
    if (mode == PTB_MODE_PATH) {
        auto shade = wf_shade_path<BVH, SMALL, STATS>;
        if ((rc = wf_smem(shade, smem_s))) return rc;
        auto extp = wf_extend_p<SMALL == PTD_FLAT ? PTD_SMALL4 : SMALL, STATS>;  // never launched for FLAT scenes
        if (persist && (rc = wf_smem(extp, smem_q))) return rc;
        const unsigned pg = persist ? pgrid(extp, smem_q, P) : 0u;
        for (int depth = 0; depth < a.max_depth; ++depth) {
            const int qi = depth & 1;
            if (persist) extp<<<pg, block, smem_q, st>>>(sc, w, depth, qi, counters, refill_thr, sm_thr_leaf);
            else ext<<<grid, block, smem_q, st>>>(sc, w, depth, qi, counters);
            shade<<<grid, block, smem_s, st>>>(sc, a, w, depth, qi);
            *launches += 2;
        }
        WF_TRY(cudaGetLastError());
    } else {
        if (persist) {
            auto extp = wf_extend_p<SMALL == PTD_FLAT ? PTD_SMALL4 : SMALL, STATS>;
            if ((rc = wf_smem(extp, smem_q))) return rc;
            extp<<<pgrid(extp, smem_q, P), block, smem_q, st>>>(sc, w, 0, 0, counters, refill_thr, sm_thr_leaf);
        } else {
            ext<<<grid, block, smem_q, st>>>(sc, w, 0, 0, counters);
        }
        WF_TRY(cudaGetLastError());
        *launches += mode == PTB_MODE_PRIMARY ? 2 : (mode == PTB_MODE_AO ? 4 : 3);
        if (mode == PTB_MODE_PRIMARY) {
            auto k = wf_shade_first<PTB_MODE_PRIMARY, BVH, SMALL, STATS>;
            if ((rc = wf_smem(k, smem_s))) return rc;
            k<<<grid, block, smem_s, st>>>(sc, a, w);
        } else if (mode == PTB_MODE_AO) {
            auto k = wf_shade_first<PTB_MODE_AO, BVH, SMALL, STATS>;
            if ((rc = wf_smem(k, smem_s))) return rc;
            k<<<grid, block, smem_s, st>>>(sc, a, w);
            const long long nr = P * a.ao_samples;
            if (persist) {
                auto shp = wf_shadow_p<PTB_MODE_AO, SMALL == PTD_FLAT ? PTD_SMALL4 : SMALL, STATS>;
                if ((rc = wf_smem(shp, smem_q))) return rc;
                shp<<<pgrid(shp, smem_q, nr), block, smem_q, st>>>(sc, a, w, (unsigned int)nr, w.work + 1, counters, refill_thr);
            } else {
                auto sh = wf_shadow<PTB_MODE_AO, BVH, SMALL, STATS>;
                if ((rc = wf_smem(sh, smem_q))) return rc;
                sh<<<(unsigned)((nr + block - 1) / block), block, smem_q, st>>>(sc, a, w, nr, counters);
            }
            wf_finish_ao<STATS><<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a, w);
        } else {
            auto k = wf_shade_first<PTB_MODE_DIRECT, BVH, SMALL, STATS>;
            if ((rc = wf_smem(k, smem_s))) return rc;
            k<<<grid, block, smem_s, st>>>(sc, a, w);
            if (persist) {
                auto shp = wf_shadow_p<PTB_MODE_DIRECT, SMALL == PTD_FLAT ? PTD_SMALL4 : SMALL, STATS>;
                if ((rc = wf_smem(shp, smem_q))) return rc;
                shp<<<pgrid(shp, smem_q, P), block, smem_q, st>>>(sc, a, w, (unsigned int)P, w.work + 1, counters, refill_thr);
            } else {
                auto sh = wf_shadow<PTB_MODE_DIRECT, BVH, SMALL, STATS>;
                if ((rc = wf_smem(sh, smem_q))) return rc;
                sh<<<grid, block, smem_q, st>>>(sc, a, w, P, counters);
            }
        }
        WF_TRY(cudaGetLastError());
    }
    if (STATS && a.stats) {
        wf_export_stats<<<(a.n_local + 255) / 256, 256, 0, st>>>(a, w);
        WF_TRY(cudaGetLastError());
        *launches += 1;
    }
    return 0;
}

// scratch layout for one batch; (re)allocates *scratch when it is too small
static int wavefront_render(cudaStream_t st, void** scratch, size_t* scratch_bytes, unsigned long long* counters,
                            int mode, const SceneDev& sc, const RenderArgs& a, bool bvh, int small, bool stats,
                            int sm_count, uint64_t* launches) {
    const size_t P = (size_t)a.frames_in_batch * a.n_local;
    const size_t n_shadow = mode == PTB_MODE_AO ? P * (size_t)a.ao_samples : (mode == PTB_MODE_DIRECT ? P : 0);
    const size_t n_counts = (size_t)a.max_depth + 2;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const bool path = mode == PTB_MODE_PATH;
    const size_t o_qo0 = take(P * 16), o_qd0 = take(P * 16), o_qm0 = take(P * 16);
    const size_t o_qo1 = take(path ? P * 16 : 0), o_qd1 = take(path ? P * 16 : 0), o_qm1 = take(path ? P * 16 : 0);
    const size_t o_hit = take(P * 16);
    const size_t o_rad = take(path ? P * 16 : 0);
    const size_t o_slotp = take(!path ? P * 16 : 0);
    const size_t o_sqw = take(n_shadow * 16);
    const size_t o_sqd = take(mode == PTB_MODE_DIRECT ? P * 16 : 0);
    const size_t o_sqc = take(mode == PTB_MODE_DIRECT ? P * 16 : 0);
    const size_t o_res = take(mode == PTB_MODE_AO ? n_shadow * 4 : 0);
    const size_t o_vis = take(mode == PTB_MODE_AO && stats ? n_shadow * 4 : 0);
    const size_t o_tst = take(mode == PTB_MODE_AO && stats ? n_shadow * 4 : 0);
    const size_t o_stats = take(stats ? P * sizeof(ptb_pixel_stats) : 0);
    const size_t o_counts = take(n_counts * 4 * 2);  // queue lengths, then work counters
    if (*scratch_bytes < off) {
        if (*scratch) WF_TRY(cudaFree(*scratch));
        *scratch = nullptr; *scratch_bytes = 0;
        WF_TRY(cudaMalloc(scratch, off));
        *scratch_bytes = off;
    }
    char* base = static_cast<char*>(*scratch);
    WfBuffers w;
    w.q_o[0] = (float4*)(base + o_qo0); w.q_d[0] = (float4*)(base + o_qd0); w.q_m[0] = (float4*)(base + o_qm0);
    w.q_o[1] = (float4*)(base + o_qo1); w.q_d[1] = (float4*)(base + o_qd1); w.q_m[1] = (float4*)(base + o_qm1);
    w.hit = (float4*)(base + o_hit);
    w.radiance = (float4*)(base + o_rad);
    w.slot_p = (float4*)(base + o_slotp);
    w.sq_w = (float4*)(base + o_sqw); w.sq_d = (float4*)(base + o_sqd); w.sq_c = (float4*)(base + o_sqc);
    w.sq_res = (int*)(base + o_res); w.sq_visits = (uint32_t*)(base + o_vis); w.sq_tests = (uint32_t*)(base + o_tst);
    w.slot_stats = (ptb_pixel_stats*)(base + o_stats);
    w.counts = (unsigned int*)(base + o_counts);
    w.work = w.counts + n_counts;
    WF_TRY(cudaMemsetAsync(w.counts, 0, n_counts * 4 * 2, st));
    if (P * (mode == PTB_MODE_AO ? (size_t)a.ao_samples : 1) >= 0xffffffffull)
        return ptb::fail(PTB_E_INVALID, "wavefront_render: batch too large for 32-bit ray indices; lower frames_per_batch");
#define WF_CASE(B, S, T) if (bvh == B && small == S && stats == T) return wf_run<B, S, T>(st, mode, sc, a, w, counters, launches, sm_count)
    if (!bvh && small == PTD_FLAT) small = PTD_SMALL4;  // brute force only needs the staged triangles
    WF_CASE(true, PTD_FLAT, false); WF_CASE(true, PTD_FLAT, true);
    WF_CASE(true, PTD_SMALL4, false); WF_CASE(true, PTD_SMALL4, true); WF_CASE(true, PTD_LARGE, false); WF_CASE(true, PTD_LARGE, true);
    WF_CASE(false, PTD_SMALL4, false); WF_CASE(false, PTD_SMALL4, true); WF_CASE(false, PTD_LARGE, false); WF_CASE(false, PTD_LARGE, true);
#undef WF_CASE
    return ptb::fail(PTB_E_INVALID, "wavefront_render: unreachable");
}

}  // namespace ptd
