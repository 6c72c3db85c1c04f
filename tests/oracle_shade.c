/* Test-side reference for render-mode samples along caller rays (ptb_scene_shade, tests/test_shade.py).
 *
 * ora_render runs the camera step (GenerateColors.cl:305-310) and then one of the oracle's per-sample integrators.  This file
 * includes the CPU oracle as it is and calls those same integrators (sample_primary, sample_ao, sample_direct, trace_rays)
 * with ray i and seed i in place of the camera's ray and post-camera seed, on a query context that walks the given tree
 * (prm->use_bvh) or loops over every triangle, as ora_render's does.  Nothing here restates the oracle's arithmetic; the test
 * builds this file into its temporary directory with the oracle's compiler flags (oracle/Makefile).
 *
 * Outputs per ray: the float4 sample (xyz as the integrator returns it, w = 1, the value ora_render's ACCUM_LINEAR writes for
 * one frame) and its ora_pixel_stats (tri_tests = the tests the sample started); counters as ora_render's.                  */
#include "oracle_pt.c"

int ora_shade(const ora_params* prm, const ora_triangle* tris, int n_tris, const ora_material* mats, const ora_bvh* bvh,
              int n_rays, const float* o, const float* d, const uint32_t* seeds, float* out, ora_pixel_stats* stats,
              ora_counters* counters) {
    if (prm->use_bvh && !bvh) return -1;
    qctr total;
    memset(&total, 0, sizeof total);
#pragma omp parallel
    {
        qctx q;
        memset(&q, 0, sizeof q);
        q.tris = tris; q.n_tris = n_tris; q.bvh = prm->use_bvh ? bvh : NULL;
#pragma omp for schedule(dynamic, 256)
        for (int i = 0; i < n_rays; i++) {
            ray_t r;
            r.o = V3(o[3 * i], o[3 * i + 1], o[3 * i + 2]);
            r.d = V3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
            uint32_t seed = seeds[i];
            sstat st;
            memset(&st, 0, sizeof st);
            uint64_t tests0 = q.c.tests;
            ora_float4 c;
            switch (prm->mode) {
                case ORA_MODE_PRIMARY: c = sample_primary(&q, mats, r, &st); break;
                case ORA_MODE_AO: c = sample_ao(&q, r, &seed, prm->ao_samples, prm->ao_max_dist, &st); break;
                case ORA_MODE_DIRECT: c = sample_direct(&q, mats, prm, r, &seed, &st); break;
                default: c = trace_rays(&q, mats, r, &seed, prm->max_depth, &st); break;
            }
            out[4 * (size_t)i] = c.x; out[4 * (size_t)i + 1] = c.y; out[4 * (size_t)i + 2] = c.z; out[4 * (size_t)i + 3] = 1.0f;
            if (stats) {
                ora_pixel_stats* ps = &stats[i];
                ps->tri = st.tri; ps->quad = st.quad; ps->t_bits = st.t_bits;
                ps->visits_primary = st.visits_primary; ps->visits_secondary = st.visits_secondary;
                ps->count = st.count; ps->id_hash = st.id_hash;
                ps->tri_tests = (uint32_t)(q.c.tests - tests0);
            }
        }
#pragma omp critical
        {
            total.closest += q.c.closest; total.any += q.c.any; total.nodes += q.c.nodes; total.tests += q.c.tests;
            total.tu += q.c.tu; total.tv += q.c.tv; total.tt += q.c.tt; total.acc += q.c.acc;
        }
    }
    if (counters) {
        counters->rays_closest = total.closest; counters->rays_any = total.any; counters->nodes = total.nodes;
        counters->tri_tests = total.tests; counters->samples = (uint64_t)n_rays;
        counters->tri_u = total.tu; counters->tri_v = total.tv; counters->tri_t = total.tt; counters->tri_accept = total.acc;
    }
    return 0;
}
