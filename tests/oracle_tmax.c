/* Test-side reference for closest-hit queries with a per-ray tmax (ptb_scene_intersect, tests/test_intersect.py).
 *
 * ora_trace's closest-hit branch always passes the reference's tmax of 1e20 (GenerateColors.cl:139).  This file includes the
 * CPU oracle as it is and calls the oracle's own traversal (bvh_query: FLAT, 4-wide or quantised binary tree) and its own
 * Moller-Trumbore test (mt_core, for the brute-force loop) with tmax[i] instead.  Nothing here restates the oracle's
 * arithmetic; the test builds this file into its temporary directory with the oracle's compiler flags (oracle/Makefile). */
#include "oracle_pt.c"

void ora_trace_closest_tmax(const ora_triangle* tris, int n_tris, const ora_bvh* bvh, int n_rays, const float* o, const float* d,
                            const float* tmax, int32_t* out_tri, float* out_t, float* out_u, float* out_v, uint32_t* out_visits,
                            uint32_t* out_tests) {
#pragma omp parallel for schedule(dynamic, 1024)
    for (int i = 0; i < n_rays; i++) {
        qctr c;
        memset(&c, 0, sizeof c);
        v3 ro = V3(o[3 * i], o[3 * i + 1], o[3 * i + 2]);
        v3 rd = V3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
        uint32_t visits = 0;
        qhit h;
        memset(&h, 0, sizeof h);
        h.tri = -1;
        int hit = 0;
        if (bvh) {
            hit = bvh_query(tris, bvh, ro, rd, tmax[i], 0, &h, &visits, &c);
        } else { /* GenerateColors.cl:137-154: ascending index, strict t < best, best starts at tmax[i] */
            float best = tmax[i];
            for (int k = 0; k < n_tris; k++) {
                float t, u, v;
                if (mt_core(ro, rd, &tris[k], &t, &u, &v, &c) && t < best) {
                    best = t;
                    h.t = t; h.u = u; h.v = v; h.tri = k;
                    hit = 1;
                }
            }
        }
        out_tri[i] = hit ? h.tri : -1;
        out_t[i] = hit ? h.t : 0.0f;
        out_u[i] = hit ? h.u : 0.0f;
        out_v[i] = hit ? h.v : 0.0f;
        out_visits[i] = visits;
        out_tests[i] = (uint32_t)c.tests;
    }
}
