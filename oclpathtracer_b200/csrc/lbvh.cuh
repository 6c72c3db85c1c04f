// lbvh.cuh -- BVH construction ON the GPU (BUILD-DEFINED; SURVEY.md 8(f).3): linear BVH by Morton order
// (Karras 2012), emitted directly in the 64-byte two-child node format the traversal kernels use.
//
//   k_lbvh_tri_bounds   per-triangle fp32 bounds + scene bounds (ordered-int atomicMin/Max)
//   k_lbvh_morton       30-bit Morton code of the box centre, key = code << 32 | triangle index (unique keys)
//   cub radix sort      64-bit keys (the only library call; the sort is not on the render path)
//   k_lbvh_topology     one thread per internal node: range + split by longest common prefix; a child whose
//                       range holds <= max_leaf triangles is emitted as a leaf reference (treelet collapse)
//   k_lbvh_fit          bottom-up: one thread per sorted triangle climbs to the root; the second arrival at a
//                       node (atomic flag) unions the two child boxes and goes on
//   k_lbvh_finish       pad the boxes, write the precomputed-edge triangle records in sorted order
//   k_scene_tris / _mats / _lights   the rest of the scene from the caller-order records: validation verdicts, edge
//                       triangles in caller order, packed materials, the light of every quad id
//
// The result is deterministic (unique sort keys, exact min/max) and equivalent to the brute-force loop by the
// same argument as the host SAH builder: every stored box is the exact bound of its triangles plus the pad.
// Quality is lower than SAH (more node visits per ray); build time is milliseconds instead of seconds.
#pragma once

#include <cub/device/device_radix_sort.cuh>

#include "host_internal.h"
#include "pt_device.cuh"

namespace ptd {

PTD_FI int float_to_ordered(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
PTD_FI float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__global__ void k_lbvh_init(int* scene_bounds) {
    if (threadIdx.x < 3) scene_bounds[threadIdx.x] = 0x7fffffff;
    else if (threadIdx.x < 6) scene_bounds[threadIdx.x] = (int)0x80000000;
}

__global__ void __launch_bounds__(256) k_lbvh_tri_bounds(const ptb_triangle* tris, int n, float4* tlo, float4* thi,
                                                         int* scene_bounds) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    if (i < n) {
        const float4* p = reinterpret_cast<const float4*>(tris + i);
        const float4 a = p[0], b = p[1], c = p[2];
        lo[0] = fminf(a.x, fminf(b.x, c.x)); hi[0] = fmaxf(a.x, fmaxf(b.x, c.x));
        lo[1] = fminf(a.y, fminf(b.y, c.y)); hi[1] = fmaxf(a.y, fmaxf(b.y, c.y));
        lo[2] = fminf(a.z, fminf(b.z, c.z)); hi[2] = fmaxf(a.z, fmaxf(b.z, c.z));
        tlo[i] = make_float4(lo[0], lo[1], lo[2], 0.f);
        thi[i] = make_float4(hi[0], hi[1], hi[2], 0.f);
    }
    for (int a = 0; a < 3; ++a) {
        int l = float_to_ordered(lo[a]), h = float_to_ordered(hi[a]);
        l = __reduce_min_sync(0xffffffffu, l);
        h = __reduce_max_sync(0xffffffffu, h);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&scene_bounds[a], l);
            atomicMax(&scene_bounds[3 + a], h);
        }
    }
}

PTD_FI unsigned int expand_bits10(unsigned int v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void __launch_bounds__(256) k_lbvh_morton(const float4* tlo, const float4* thi, int n, const int* scene_bounds,
                                                     unsigned long long* keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 lo = tlo[i], hi = thi[i];
    const float c[3] = {0.5f * lo.x + 0.5f * hi.x, 0.5f * lo.y + 0.5f * hi.y, 0.5f * lo.z + 0.5f * hi.z};
    unsigned int q[3];
    for (int a = 0; a < 3; ++a) {
        const float smin = ordered_to_float(scene_bounds[a]), smax = ordered_to_float(scene_bounds[3 + a]);
        const float ext = smax - smin;
        float t = ext > 0.f ? (c[a] - smin) / ext : 0.f;
        t = fminf(fmaxf(t * 1024.0f, 0.0f), 1023.0f);
        q[a] = (unsigned int)t;
    }
    const unsigned int code = (expand_bits10(q[0]) << 2) | (expand_bits10(q[1]) << 1) | expand_bits10(q[2]);
    keys[i] = ((unsigned long long)code << 32) | (unsigned int)i;
}

PTD_FI int lbvh_delta(const unsigned long long* keys, int n, int a, int b) {
    if (b < 0 || b >= n) return -1;
    return __clzll((long long)(keys[a] ^ keys[b]));
}

// one thread per internal node (Karras 2012, fig. 4).  parent[] covers internal nodes [0,n-1) then leaves [n-1, 2n-1).
__global__ void __launch_bounds__(256) k_lbvh_topology(const unsigned long long* keys, int n, int max_leaf, float4* nodes,
                                                       int* parent) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int dmin = lbvh_delta(keys, n, i, i - d);
    int lmax = 2;
    while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = lbvh_delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) / 2;; t = (t + 1) / 2) {
        if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int gamma = i + s * d + (d < 0 ? d : 0);
    const int first = i < j ? i : j, last = i < j ? j : i;
    // children: [first, gamma] and [gamma+1, last]
    const int nl = gamma - first + 1, nr = last - gamma;
    const int left = nl <= max_leaf ? PTB_BVH_LEAF_REF(first, nl) : gamma;
    const int right = nr <= max_leaf ? PTB_BVH_LEAF_REF(gamma + 1, nr) : gamma + 1;
    nodes[4 * (size_t)i + 0].w = __int_as_float(left);
    nodes[4 * (size_t)i + 1].w = __int_as_float(right);
    // parents for the bottom-up pass use the UNcollapsed topology (every Karras node gets its box)
    if (first == gamma) parent[(n - 1) + gamma] = (i << 1) | 0; else parent[gamma] = (i << 1) | 0;
    if (last == gamma + 1) parent[(n - 1) + gamma + 1] = (i << 1) | 1; else parent[gamma + 1] = (i << 1) | 1;
    if (i == 0) parent[0] = -1;
}

__global__ void __launch_bounds__(256) k_lbvh_fit(const unsigned long long* keys, const float4* tlo, const float4* thi, int n,
                                                  float4* nodes, const int* parent, int* flags, int* max_depth) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int tri = (int)(keys[k] & 0xffffffffull);
    float4 lo = tlo[tri], hi = thi[tri];
    int p = parent[(n - 1) + k];
    int depth = 0;  // internal nodes on the longest path down from the subtree this thread carries (0 at a leaf)
    while (p >= 0) {
        const int node = p >> 1, side = p & 1;
        float4* nd = nodes + 4 * (size_t)node;
        // keep the child reference stored in .w of words 0/1
        if (side == 0) {
            nd[0].x = lo.x; nd[0].y = lo.y; nd[0].z = lo.z;
            nd[1].x = hi.x; nd[1].y = hi.y; nd[1].z = hi.z;
        } else {
            nd[2] = make_float4(lo.x, lo.y, lo.z, 0.f);
            nd[3] = make_float4(hi.x, hi.y, hi.z, 0.f);
        }
        __threadfence();
        // the first arrival leaves its subtree's depth + 1 and stops (the sibling subtree is not finished yet); the second
        // takes the deeper of the two, so the root gets the tree's depth whichever leaves' threads climb to it
        const int sibling = atomicAdd(&flags[node], depth + 1);
        if (sibling == 0) return;
        depth = 1 + max(depth, sibling - 1);
        __threadfence();
        const float4 a0 = __ldcg(nd), a1 = __ldcg(nd + 1), b0 = __ldcg(nd + 2), b1 = __ldcg(nd + 3);  // L2, not a stale L1 line
        lo = make_float4(fminf(a0.x, b0.x), fminf(a0.y, b0.y), fminf(a0.z, b0.z), 0.f);
        hi = make_float4(fmaxf(a1.x, b1.x), fmaxf(a1.y, b1.y), fmaxf(a1.z, b1.z), 0.f);
        p = parent[node];
    }
    atomicMax(max_depth, depth);
}

__global__ void __launch_bounds__(256) k_lbvh_finish(const ptb_triangle* tris, const unsigned long long* keys, int n, float pad_rel,
                                                     const int* scene_bounds, float4* nodes, float4* otris, int* tri_order) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float dx = ordered_to_float(scene_bounds[3]) - ordered_to_float(scene_bounds[0]);
    const float dy = ordered_to_float(scene_bounds[4]) - ordered_to_float(scene_bounds[1]);
    const float dz = ordered_to_float(scene_bounds[5]) - ordered_to_float(scene_bounds[2]);
    const float pad = pad_rel * sqrtf(dx * dx + dy * dy + dz * dz);  // pad_rel > 0: checked by the scene constructors
    if (i < n - 1) {
        float4* nd = nodes + 4 * (size_t)i;
        // padded [lo, hi] of each child -> centre / half-extent widened by two ulps (same rule as the host builder)
        float4 a = nd[0], b = nd[1], c = nd[2], d = nd[3];
        auto ce = [pad](float lo, float hi, float& cc, float& ee) {
            lo -= pad; hi += pad;
            cc = 0.5f * lo + 0.5f * hi;
            const float h = 0.5f * hi - 0.5f * lo;
            ee = h + 2.4e-7f * (fabsf(cc) + h);
        };
        float4 o0 = a, o1 = b, o2 = c, o3 = d;
        ce(a.x, b.x, o0.x, o1.x); ce(a.y, b.y, o0.y, o1.y); ce(a.z, b.z, o0.z, o1.z);
        ce(c.x, d.x, o2.x, o3.x); ce(c.y, d.y, o2.y, o3.y); ce(c.z, d.z, o2.z, o3.z);
        o2.w = 0.f; o3.w = 0.f;
        nd[0] = o0; nd[1] = o1; nd[2] = o2; nd[3] = o3;
    }
    if (i < n) {
        const int tri = (int)(keys[i] & 0xffffffffull);
        const float4* p = reinterpret_cast<const float4*>(tris + tri);
        const float4 p1 = p[0], p2 = p[1], p3 = p[2];
        const int quad = reinterpret_cast<const int*>(tris + tri)[12];
        otris[3 * (size_t)i + 0] = make_float4(p1.x, p1.y, p1.z, __int_as_float(tri));
        otris[3 * (size_t)i + 1] = make_float4(p2.x - p1.x, p2.y - p1.y, p2.z - p1.z, __int_as_float(quad));  // GenerateColors.cl:92
        otris[3 * (size_t)i + 2] = make_float4(p3.x - p1.x, p3.y - p1.y, p3.z - p1.z, 0.f);                   // GenerateColors.cl:93
        tri_order[i] = tri;
    }
}

// ---- the rest of a device-built scene, from the caller-order records on the device ------------------------------------
// (ptb_scene_create_gpu, ptb_scene_create_from_device).  Every output is a bit copy or a plain fp32 subtraction of the records,
// so it equals what the host computes from the same records (make_edge_tris, the material packing of scene_create_impl,
// ptb_light_from_quad).

// The area light of one quad id as ptb_light_from_quad derives it; q = the first even triangle index with q + 1 < n and
// id == quad, or a value >= n when there is no such pair (the table starts as 0x7f bytes).
struct SceneLight {
    int32_t q;
    float p1[3], ea[3], eb[3];
};
static_assert(sizeof(SceneLight) == 40, "SceneLight is read back as 40-byte records");

// One thread per triangle: the validation verdicts (bad[0]: the lowest index whose id is outside [0, n_mats), as
// index << 32 | id bits; bad[1]: the lowest index with a vertex float failing |v| <= 3e38, w included; both start all ones),
// the caller-order edge triangle (edge_tri: index = i, quad = id, pad = 0) and the first even q of each quad id.
__global__ void __launch_bounds__(256) k_scene_tris(const ptb_triangle* tris, int n, int n_mats, unsigned long long* bad,
                                                    float4* otris, SceneLight* lights) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool bad_id = false, bad_v = false;
    int id = -1;
    if (i < n) {
        const float4* p = reinterpret_cast<const float4*>(tris + i);
        const float4 a = p[0], b = p[1], c = p[2];
        id = reinterpret_cast<const int*>(tris + i)[12];
        bad_id = id < 0 || id >= n_mats;
        const float v[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
        for (int k = 0; k < 12; ++k) bad_v |= !(fabsf(v[k]) <= 3.0e38f);
        otris[3 * (size_t)i + 0] = make_float4(a.x, a.y, a.z, __int_as_float(i));
        otris[3 * (size_t)i + 1] = make_float4(b.x - a.x, b.y - a.y, b.z - a.z, __int_as_float(id));  // GenerateColors.cl:92
        otris[3 * (size_t)i + 2] = make_float4(c.x - a.x, c.y - a.y, c.z - a.z, 0.f);                  // GenerateColors.cl:93
    }
    // lanes hold consecutive indices: the lowest offending lane of a warp has the warp's lowest index, one atomic per warp
    const unsigned mid = __ballot_sync(0xffffffffu, bad_id), mv = __ballot_sync(0xffffffffu, bad_v);
    if (mid && lane == __ffs(mid) - 1) atomicMin(&bad[0], ((unsigned long long)i << 32) | (unsigned int)id);
    if (mv && lane == __ffs(mv) - 1) atomicMin(&bad[1], (unsigned long long)i);
    // light pairs: lanes of one id meet in one atomic (tessellated scenes hold long runs of one id)
    const int key = (i < n && (i & 1) == 0 && i + 1 < n && !bad_id) ? id : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(peers) - 1) atomicMin(&lights[key].q, i);
}

// one thread per material: the two float4s the kernels read (albedo.xyz, roughness | emissive.xyz, bits of type)
__global__ void __launch_bounds__(256) k_scene_mats(const ptb_material* mats, int n_mats, float4* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_mats) return;
    const float4* p = reinterpret_cast<const float4*>(mats + i);
    const float4 albedo = p[0], emissive = p[1], rt = p[2];  // rt.x = roughness, rt.y = type
    out[2 * (size_t)i] = make_float4(albedo.x, albedo.y, albedo.z, rt.x);
    out[2 * (size_t)i + 1] = make_float4(emissive.x, emissive.y, emissive.z, rt.y);
}

// one thread per quad id, after k_scene_tris: p1 = tris[q].p1, ea = tris[q].p2 - p1, eb = tris[q + 1].p2 - p1
__global__ void __launch_bounds__(256) k_scene_lights(const ptb_triangle* tris, int n, int n_mats, SceneLight* lights) {
    const int quad = blockIdx.x * blockDim.x + threadIdx.x;
    if (quad >= n_mats) return;
    SceneLight& L = lights[quad];
    const int q = L.q;
    if (q >= n) return;
    const float4 a = reinterpret_cast<const float4*>(tris + q)[0], b = reinterpret_cast<const float4*>(tris + q)[1];
    const float4 d = reinterpret_cast<const float4*>(tris + q + 1)[1];
    L.p1[0] = a.x; L.p1[1] = a.y; L.p1[2] = a.z;
    L.ea[0] = b.x - a.x; L.ea[1] = b.y - a.y; L.ea[2] = b.z - a.z;
    L.eb[0] = d.x - a.x; L.eb[1] = d.y - a.y; L.eb[2] = d.z - a.z;
}

#define LBVH_TRY(expr)                                                                                       \
    do {                                                                                                     \
        cudaError_t e__ = (expr);                                                                            \
        if (e__ != cudaSuccess) { rc = ptb::fail(PTB_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); goto cleanup; } \
    } while (0)

// d_tris: n caller-order records on the device.  Outputs are cudaMalloc'd here (caller frees).  The `readback` bytes at
// d_readback (work the caller enqueued before on `st`) are copied to h_readback in the same synchronisation as the depth.
static int build_lbvh_device(cudaStream_t st, const ptb_triangle* d_tris, int n, int max_leaf, float pad_rel, float4** d_nodes_out,
                             float4** d_otris_out, int** d_order_out, int* depth_out, const void* d_readback, void* h_readback,
                             size_t readback) {
    int rc = PTB_OK;
    float4 *tlo = nullptr, *thi = nullptr, *nodes = nullptr, *otris = nullptr;
    unsigned long long *keys = nullptr, *keys_sorted = nullptr;
    int *parent = nullptr, *flags = nullptr, *misc = nullptr, *order = nullptr;
    void* temp = nullptr;
    size_t temp_bytes = 0;
    const int grid_n = (n + 255) / 256;
    int depth = 0;
    if (n < 2) return ptb::fail(PTB_E_INVALID, "build_lbvh_device: needs at least two triangles");
    if (max_leaf < 1) max_leaf = 1;
    if (max_leaf > PTB_BVH_MAX_LEAF) max_leaf = PTB_BVH_MAX_LEAF;
    LBVH_TRY(cudaMalloc((void**)&tlo, sizeof(float4) * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&thi, sizeof(float4) * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&keys, 8 * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&keys_sorted, 8 * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&parent, 4 * (size_t)(2 * n)));
    LBVH_TRY(cudaMalloc((void**)&flags, 4 * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&misc, 4 * 8));
    LBVH_TRY(cudaMalloc((void**)&nodes, 64 * (size_t)(n - 1)));
    LBVH_TRY(cudaMalloc((void**)&otris, 48 * (size_t)n));
    LBVH_TRY(cudaMalloc((void**)&order, 4 * (size_t)n));
    LBVH_TRY(cudaMemsetAsync(flags, 0, 4 * (size_t)n, st));
    LBVH_TRY(cudaMemsetAsync(misc, 0, 32, st));
    k_lbvh_init<<<1, 32, 0, st>>>(misc);
    k_lbvh_tri_bounds<<<grid_n, 256, 0, st>>>(d_tris, n, tlo, thi, misc);
    k_lbvh_morton<<<grid_n, 256, 0, st>>>(tlo, thi, n, misc, keys);
    LBVH_TRY(cudaGetLastError());
    LBVH_TRY(cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, keys, keys_sorted, n, 0, 64, st));
    LBVH_TRY(cudaMalloc(&temp, temp_bytes));
    LBVH_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys, keys_sorted, n, 0, 64, st));
    k_lbvh_topology<<<(n - 1 + 255) / 256, 256, 0, st>>>(keys_sorted, n, max_leaf, nodes, parent);
    k_lbvh_fit<<<grid_n, 256, 0, st>>>(keys_sorted, tlo, thi, n, nodes, parent, flags, misc + 6);
    k_lbvh_finish<<<grid_n, 256, 0, st>>>(d_tris, keys_sorted, n, pad_rel, misc, nodes, otris, order);
    LBVH_TRY(cudaGetLastError());
    LBVH_TRY(cudaMemcpyAsync(&depth, misc + 6, 4, cudaMemcpyDeviceToHost, st));
    if (readback) LBVH_TRY(cudaMemcpyAsync(h_readback, d_readback, readback, cudaMemcpyDeviceToHost, st));
    LBVH_TRY(cudaStreamSynchronize(st));
    *d_nodes_out = nodes; *d_otris_out = otris; *d_order_out = order; *depth_out = depth;
    nodes = nullptr; otris = nullptr; order = nullptr;
cleanup:
    for (void* p : {(void*)tlo, (void*)thi, (void*)keys, (void*)keys_sorted, (void*)parent, (void*)flags, (void*)misc, temp,
                    (void*)nodes, (void*)otris, (void*)order})
        if (p) cudaFree(p);
    return rc;
}

// ---- quantised encoding of a binary tree (ptb_bvh_nodeq; DESIGN.md section 4 "Quantised binary nodes") ----------------
// A pure function of the fp32 node array, evaluated on the device for host-built and device-built trees alike; the CPU
// oracle re-states it (ora_bvh_quantize, rules Q1-Q3) and the tests compare the bytes.  IEEE double, no
// contraction (--fmad=false).
// grid[0..2] = q_lo, grid[3..5] = q_step from the ROOT's child boxes (rule Q1)
__global__ void k_quant_grid(const float4* nodes, float* grid) {
    if (blockIdx.x || threadIdx.x) return;
    const float4 n0 = nodes[0], n1 = nodes[1], n2 = nodes[2], n3 = nodes[3];
    const float c[2][3] = {{n0.x, n0.y, n0.z}, {n2.x, n2.y, n2.z}};
    const float e[2][3] = {{n1.x, n1.y, n1.z}, {n3.x, n3.y, n3.z}};
    const int refs[2] = {__float_as_int(n0.w), __float_as_int(n1.w)};
    for (int a = 0; a < 3; ++a) {
        double lo = 0.0, hi = 0.0;
        bool have = false;
        for (int k = 0; k < 2; ++k) {
            if (refs[k] == PTB_BVH_EMPTY) continue;
            const double l = (double)c[k][a] - (double)e[k][a], h = (double)c[k][a] + (double)e[k][a];
            if (!have || l < lo) lo = l;
            if (!have || h > hi) hi = h;
            have = true;
        }
        double ext = hi - lo;
        if (!(ext > 0.0)) ext = 1.0;
        const double margin = ext / 1024.0;
        grid[a] = (float)(lo - margin);
        grid[3 + a] = (float)((ext + 2.0 * margin) / 65000.0);
    }
}
// rules Q2, Q3: one thread per node
__global__ void __launch_bounds__(256) k_quant_nodes(const float4* nodes, int n_nodes, const float* grid, uint4* q) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const float4 n0 = nodes[4 * (size_t)i], n1 = nodes[4 * (size_t)i + 1], n2 = nodes[4 * (size_t)i + 2], n3 = nodes[4 * (size_t)i + 3];
    const float c[2][3] = {{n0.x, n0.y, n0.z}, {n2.x, n2.y, n2.z}};
    const float e[2][3] = {{n1.x, n1.y, n1.z}, {n3.x, n3.y, n3.z}};
    const int refs[2] = {__float_as_int(n0.w), __float_as_int(n1.w)};
    uint32_t w[6];
    for (int k = 0; k < 2; ++k)
        for (int a = 0; a < 3; ++a) {
            uint32_t ql = 65535u, qh = 0u;
            if (refs[k] != PTB_BVH_EMPTY) {
                const double plo = (double)c[k][a] - (double)e[k][a], phi = (double)c[k][a] + (double)e[k][a];
                const double fl = floor((plo - (double)grid[a]) / (double)grid[3 + a]) - 1.0;
                const double fh = ceil((phi - (double)grid[a]) / (double)grid[3 + a]) + 1.0;
                ql = fl < 0.0 ? 0u : fl > 65535.0 ? 65535u : (uint32_t)(long long)fl;
                qh = fh < 0.0 ? 0u : fh > 65535.0 ? 65535u : (uint32_t)(long long)fh;
            }
            w[3 * k + a] = ql | (qh << 16);
        }
    q[2 * (size_t)i] = make_uint4(w[0], w[1], w[2], w[3]);
    q[2 * (size_t)i + 1] = make_uint4(w[4], w[5], (uint32_t)refs[0], (uint32_t)refs[1]);
}

}  // namespace ptd
