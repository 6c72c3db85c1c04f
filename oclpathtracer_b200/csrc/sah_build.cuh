// sah_build.cuh -- the host's binned-SAH tree (bvh_build.cpp, Builder::build) built ON the device, byte for byte
// (ptb_bvh_params.builder = PTB_BUILDER_SAH; DESIGN.md section 4 "Device SAH builder").
//
// The host tree is a pure function of sets of triangles: node and centroid bounds are exact min/max, bin counts are exact,
// the sweep reads only those, a partition is a set split, the median fallback cuts the set at its n/2 smallest caller
// indices and a leaf lists its triangles by caller index.  A leaf over [b, e) starts at b, and the final numbering depends on
// the topology only.  So the device evaluates the same expressions in the same precision (IEEE double sweep, no contraction)
// and may use any partition order and schedule.  Every range's index list is kept ascending in caller index: the root is
// 0..n-1 and every partition is stable, so the median fallback is a cut at n/2 and leaves need no sort.
//
//   k_lbvh_tri_bounds   per-triangle bounds and the scene bounds (shared with the LBVH)
//   ranges of more than SAH_T primitives, level by level, each range tiled over CTAs of SAH_TILE primitives:
//     k_sah_plan        tile table of the level's ranges
//     k_sah_bounds      exact box and centroid bounds of each range
//     k_sah_bin         per axis and bin: box and count, privatised in shared memory, merged with integer atomics
//     k_sah_decide      one warp per range: the host's sweep, the split, the node record, the child ranges
//     k_sah_count, cub scan, k_sah_scatter   stable partition into the other index buffer
//   k_sah_small         one CTA per range of <= SAH_T primitives: its whole subtree by the same rules, in shared memory
//   k_sah_keys, cub scan + sort, k_sah_queue, k_sah_newid, k_sah_emit, k_sah_tris   renumbering (breadth-first prefix of
//                       smem_nodes nodes, then depth-first subtrees in the host queue's order) and the output records
//
// Min/max are integer atomics on order-preserving keys of the floats, never float atomics, so nothing depends on arrival
// order.  An internal node over [b, e) split at mid takes the temporary id mid - 1: split positions are unique, so ids need no
// counter and fit n - 1 slots.
#pragma once

#include <climits>

#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "lbvh.cuh"

namespace ptd {

constexpr int SAH_T = 1024;             // ranges above this many primitives take the level-synchronous path
constexpr int SAH_TILE = 2048;          // primitives per CTA in the large-range passes
constexpr int SAH_SMALL_THREADS = 256;  // k_sah_small
constexpr int SAH_BIN_WORDS = 7;        // per bin: ~key(lo) xyz, key(hi) xyz, count

struct SahParams {
    int max_leaf, n_bins;
    double k_traverse;  // Builder::kTraverse: traverse_cost if > 0, else 1.2
};

struct SahTask {
    int b, e;
    int parent;         // temporary id * 2 + side of the slot that references this range; -1: the root
    int level;          // root = 1
    int lanc;           // ancestors that hold this range in their child0 subtree
    int buf;            // index buffer holding the range
    int axis, split;    // k_sah_decide: SAH split (axis < 0: cut at n / 2)
    int mid;
    float cmin, scale;
};

// order-preserving unsigned key of a float: max of keys = max of floats, max of ~keys = min (both start at 0)
PTD_FI unsigned sah_key(float f) { return (unsigned)float_to_ordered(f) ^ 0x80000000u; }
PTD_FI float sah_unkey(unsigned u) { return ordered_to_float((int)(u ^ 0x80000000u)); }

// Builder::bin_of.  x86 hosts convert with cvttss2si, which gives INT_MIN for NaN and out-of-range values (bin 0); the
// device conversion saturates, so it is told apart here.  Reached only through a centroid extent so small that the scale
// overflows, or records the validation refuses.
PTD_FI int sah_bin(float c, float cmin, float scale, int nb) {
    const float x = (c - cmin) * scale;
#if defined(__x86_64__) || defined(__i386__)
    const int k = (x >= -2147483648.0f && x < 2147483648.0f) ? (int)x : INT_MIN;
#else
    const int k = (int)x;
#endif
    return k < 0 ? 0 : (k >= nb ? nb - 1 : k);
}

// Box::half_area, in double
PTD_FI double sah_half_area(const float lo[3], const float hi[3]) {
    const double dx = double(hi[0]) - lo[0], dy = double(hi[1]) - lo[1], dz = double(hi[2]) - lo[2];
    return dx * dy + dy * dz + dz * dx;
}

// Box::grow with std::min / std::max semantics, from a bin's words
PTD_FI void sah_grow(float lo[3], float hi[3], const unsigned* w) {
    for (int a = 0; a < 3; ++a) {
        const float l = sah_unkey(~w[a]), h = sah_unkey(w[3 + a]);
        lo[a] = l < lo[a] ? l : lo[a];
        hi[a] = hi[a] < h ? h : hi[a];
    }
}

// The sweep of one axis in Builder::build: the first strictly lowest cost over the splits between bins k-1 and k, k = 1..nb-1.
// bins: [nb][SAH_BIN_WORDS].  best_cost stays INFINITY when no boundary separates the set.
__device__ __noinline__ void sah_sweep(const unsigned* bins, int nb, double& best_cost, int& best_split) {
    double right_area[256];
    int right_cnt[256];
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    int cnt = 0;
    for (int k = nb - 1; k >= 1; --k) {
        const unsigned* w = bins + k * SAH_BIN_WORDS;
        if (w[6]) sah_grow(lo, hi, w);
        cnt += (int)w[6];
        right_area[k] = cnt ? sah_half_area(lo, hi) : 0.0;
        right_cnt[k] = cnt;
    }
    for (int a = 0; a < 3; ++a) { lo[a] = INFINITY; hi[a] = -INFINITY; }
    cnt = 0;
    best_cost = INFINITY;
    best_split = -1;
    for (int k = 1; k < nb; ++k) {
        const unsigned* w = bins + (k - 1) * SAH_BIN_WORDS;
        if (w[6]) sah_grow(lo, hi, w);
        cnt += (int)w[6];
        if (cnt == 0 || right_cnt[k] == 0) continue;
        const double cost = sah_half_area(lo, hi) * cnt + right_area[k] * right_cnt[k];
        if (cost < best_cost) { best_cost = cost; best_split = k; }
    }
}

// the leaf test of Builder::build
PTD_FI bool sah_leaf(int n, bool force_split, int best_axis, double best_cost, double parent_area, const SahParams& p) {
    const double split_cost = (best_axis >= 0 && parent_area > 0.0) ? p.k_traverse + 1.0 * best_cost / parent_area
                                                                    : (best_axis >= 0 ? p.k_traverse : INFINITY);
    const bool can_leaf = n <= p.max_leaf && !force_split;
    return n == 1 || (can_leaf && double(n) * 1.0 <= split_cost);
}

// The per-range accumulator: 12 words, ~key(lo) xyz, key(hi) xyz, ~key(centroid lo) xyz, key(centroid hi) xyz
PTD_FI void sah_acc_prim(unsigned acc[12], float4 l, float4 h) {
    const float lo[3] = {l.x, l.y, l.z}, hi[3] = {h.x, h.y, h.z};
    for (int a = 0; a < 3; ++a) {
        const float c = 0.5f * lo[a] + 0.5f * hi[a];  // Prim::c
        acc[a] = max(acc[a], ~sah_key(lo[a]));
        acc[3 + a] = max(acc[3 + a], sah_key(hi[a]));
        acc[6 + a] = max(acc[6 + a], ~sah_key(c));
        acc[9 + a] = max(acc[9 + a], sah_key(c));
    }
}
PTD_FI void sah_decode(const unsigned* w, float lo[3], float hi[3], float clo[3], float chi[3]) {
    for (int a = 0; a < 3; ++a) {
        lo[a] = sah_unkey(~w[a]); hi[a] = sah_unkey(w[3 + a]);
        clo[a] = sah_unkey(~w[6 + a]); chi[a] = sah_unkey(w[9 + a]);
    }
}

// Temporary node records, indexed by temporary id: child references, exact child boxes, [b, e), level, lanc
struct SahTmp {
    int2* child;
    float4* box;   // 4 per node: lo0, hi0, lo1, hi1
    int4* info;    // b, e, level, lanc
    int* used;     // 1 for every id that is a node
    int* root_id;
    int* max_level;
};

// the node or leaf `ref` over exact bounds lo/hi becomes child `side` of its parent (or the root)
PTD_FI void sah_link(const SahTmp& t, int parent, int ref, const float lo[3], const float hi[3]) {
    if (parent < 0) { *t.root_id = ref; return; }
    const int node = parent >> 1, side = parent & 1;
    t.box[4 * (size_t)node + 2 * side] = make_float4(lo[0], lo[1], lo[2], 0.f);
    t.box[4 * (size_t)node + 2 * side + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
    if (side == 0) t.child[node].x = ref; else t.child[node].y = ref;
}
PTD_FI void sah_node(const SahTmp& t, int id, int b, int e, int level, int lanc) {
    t.info[id] = make_int4(b, e, level, lanc);
    t.used[id] = 1;
    atomicMax(t.max_level, level);
}

PTD_FI float sah_pick(float4 v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }

// ---- ranges of more than SAH_T primitives ------------------------------------------------------------------------------

// last task whose first tile is <= x
PTD_FI int sah_tile_task(const int* tile_start, int n_tasks, int x) {
    int lo = 0, hi = n_tasks - 1;
    while (lo < hi) {
        const int m = (lo + hi + 1) >> 1;
        if (tile_start[m] <= x) lo = m; else hi = m - 1;
    }
    return lo;
}

// tile_start[t] = first tile of task t, tile_start[n_tasks] = the level's tile count
__global__ void __launch_bounds__(1024) k_sah_plan(const SahTask* tasks, const int* n_tasks_p, int* tile_start) {
    using Scan = cub::BlockScan<int, 1024>;
    __shared__ typename Scan::TempStorage ts;
    __shared__ int carry;
    const int nt = *n_tasks_p;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nt; base += 1024) {
        const int t = base + threadIdx.x;
        const int tiles = t < nt ? (tasks[t].e - tasks[t].b + SAH_TILE - 1) / SAH_TILE : 0;
        int excl, total;
        Scan(ts).ExclusiveSum(tiles, excl, total);
        if (t < nt) tile_start[t] = carry + excl;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_start[nt] = carry;
}

struct SahTile {
    int t, j0, j1;
};
PTD_FI bool sah_tile(const SahTask* tasks, const int* n_tasks_p, const int* tile_start, SahTile& out) {
    const int nt = *n_tasks_p, x = blockIdx.x;
    if (x >= tile_start[nt]) return false;
    out.t = sah_tile_task(tile_start, nt, x);
    out.j0 = tasks[out.t].b + (x - tile_start[out.t]) * SAH_TILE;
    out.j1 = min(tasks[out.t].e, out.j0 + SAH_TILE);
    return true;
}

// exact box and centroid bounds of every range (tb: 12 words per task, zeroed)
__global__ void __launch_bounds__(256) k_sah_bounds(const SahTask* tasks, const int* n_tasks_p, const int* tile_start,
                                                    const int* idx0, const int* idx1, const float4* tlo, const float4* thi,
                                                    unsigned* tb) {
    SahTile tl;
    if (!sah_tile(tasks, n_tasks_p, tile_start, tl)) return;
    const int* src = tasks[tl.t].buf ? idx1 : idx0;
    __shared__ unsigned red[12];
    if (threadIdx.x < 12) red[threadIdx.x] = 0;
    unsigned acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = tl.j0 + threadIdx.x; j < tl.j1; j += blockDim.x) {
        const int i = src[j];
        sah_acc_prim(acc, tlo[i], thi[i]);
    }
    __syncthreads();
    for (int k = 0; k < 12; ++k) {
        const unsigned v = __reduce_max_sync(0xffffffffu, acc[k]);
        if ((threadIdx.x & 31) == 0) atomicMax(&red[k], v);
    }
    __syncthreads();
    if (threadIdx.x < 12) atomicMax(&tb[12 * (size_t)tl.t + threadIdx.x], red[threadIdx.x]);
}

// per axis with a nonzero centroid extent: the host's bins (bins: [task][3][nb][SAH_BIN_WORDS], zeroed)
__global__ void __launch_bounds__(256) k_sah_bin(const SahTask* tasks, const int* n_tasks_p, const int* tile_start, const int* idx0,
                                                 const int* idx1, const float4* tlo, const float4* thi, const unsigned* tb, int nb,
                                                 unsigned* bins) {
    SahTile tl;
    if (!sah_tile(tasks, n_tasks_p, tile_start, tl)) return;
    __shared__ unsigned sb[3 * 256 * SAH_BIN_WORDS];
    const int* src = tasks[tl.t].buf ? idx1 : idx0;
    float lo[3], hi[3], clo[3], chi[3], scale[3];
    sah_decode(tb + 12 * (size_t)tl.t, lo, hi, clo, chi);
    bool on[3];
    for (int a = 0; a < 3; ++a) {
        on[a] = chi[a] > clo[a];
        scale[a] = on[a] ? float(nb) / (chi[a] - clo[a]) : 0.f;
    }
    for (int k = threadIdx.x; k < 3 * nb * SAH_BIN_WORDS; k += blockDim.x) sb[k] = 0;
    __syncthreads();
    for (int j = tl.j0 + threadIdx.x; j < tl.j1; j += blockDim.x) {
        const int i = src[j];
        const float4 l = tlo[i], h = thi[i];
        const unsigned kl[3] = {~sah_key(l.x), ~sah_key(l.y), ~sah_key(l.z)}, kh[3] = {sah_key(h.x), sah_key(h.y), sah_key(h.z)};
        for (int a = 0; a < 3; ++a) {
            if (!on[a]) continue;
            const float c = 0.5f * sah_pick(l, a) + 0.5f * sah_pick(h, a);
            unsigned* w = sb + (a * nb + sah_bin(c, clo[a], scale[a], nb)) * SAH_BIN_WORDS;
            for (int d = 0; d < 3; ++d) { atomicMax(&w[d], kl[d]); atomicMax(&w[3 + d], kh[d]); }
            atomicAdd(&w[6], 1u);
        }
    }
    __syncthreads();
    unsigned* g = bins + (size_t)tl.t * 3 * nb * SAH_BIN_WORDS;
    for (int k = threadIdx.x; k < 3 * nb; k += blockDim.x) {
        const unsigned* w = sb + k * SAH_BIN_WORDS;
        if (!w[6]) continue;
        for (int d = 0; d < 6; ++d) atomicMax(&g[k * SAH_BIN_WORDS + d], w[d]);
        atomicAdd(&g[k * SAH_BIN_WORDS + 6], w[6]);
    }
}

// One warp per range: lanes 0..2 sweep x, y, z; lane 0 takes the first strictly lowest, records the node (a range of more
// than SAH_T >= PTB_BVH_MAX_LEAF primitives is never a leaf) and queues the two child ranges.
__global__ void __launch_bounds__(128) k_sah_decide(SahTask* tasks, const int* n_tasks_p, const unsigned* tb, const unsigned* bins,
                                                    SahParams p, SahTmp tmp, SahTask* next, int* n_next, SahTask* small, int* n_small) {
    const int t = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (t >= *n_tasks_p) return;  // whole warps
    const int nb = p.n_bins;
    float lo[3], hi[3], clo[3], chi[3];
    sah_decode(tb + 12 * (size_t)t, lo, hi, clo, chi);
    double cost = INFINITY;
    int split = -1;
    if (lane < 3 && chi[lane] > clo[lane]) sah_sweep(bins + ((size_t)t * 3 + lane) * nb * SAH_BIN_WORDS, nb, cost, split);
    const double c1 = __shfl_sync(0xffffffffu, cost, 1), c2 = __shfl_sync(0xffffffffu, cost, 2);
    const int s1 = __shfl_sync(0xffffffffu, split, 1), s2 = __shfl_sync(0xffffffffu, split, 2);
    if (lane) return;
    int axis = -1;
    double best = INFINITY;
    const double cs[3] = {cost, c1, c2};
    const int ss[3] = {split, s1, s2};
    for (int a = 0; a < 3; ++a)
        if (cs[a] < best) { best = cs[a]; axis = a; split = ss[a]; }
    SahTask T = tasks[t];
    const int n = T.e - T.b;
    int left = n / 2;
    if (axis >= 0) {
        left = 0;
        const unsigned* w = bins + ((size_t)t * 3 + axis) * nb * SAH_BIN_WORDS;
        for (int k = 0; k < split; ++k) left += (int)w[k * SAH_BIN_WORDS + 6];
        T.cmin = clo[axis];
        T.scale = float(nb) / (chi[axis] - clo[axis]);
    }
    T.axis = axis; T.split = split; T.mid = T.b + left;
    tasks[t] = T;
    const int id = T.mid - 1;
    sah_node(tmp, id, T.b, T.e, T.level, T.lanc);
    sah_link(tmp, T.parent, id, lo, hi);
    for (int side = 0; side < 2; ++side) {
        SahTask c{};
        c.b = side ? T.mid : T.b; c.e = side ? T.e : T.mid;
        c.parent = 2 * id + side; c.level = T.level + 1; c.lanc = T.lanc + (side == 0); c.buf = T.buf ^ 1;
        if (c.e - c.b > SAH_T) next[atomicAdd(n_next, 1)] = c;
        else small[atomicAdd(n_small, 1)] = c;
    }
}

PTD_FI bool sah_goes_left(const SahTask& T, int j, float4 l, float4 h, int nb) {
    if (T.axis < 0) return j - T.b < (T.e - T.b) / 2;
    const float c = 0.5f * sah_pick(l, T.axis) + 0.5f * sah_pick(h, T.axis);
    return sah_bin(c, T.cmin, T.scale, nb) < T.split;
}

// left primitives per tile (0 for the grid's spare CTAs, so the scan may run over the whole grid)
__global__ void __launch_bounds__(256) k_sah_count(const SahTask* tasks, const int* n_tasks_p, const int* tile_start, const int* idx0,
                                                   const int* idx1, const float4* tlo, const float4* thi, int nb, int* tile_left) {
    SahTile tl;
    if (!sah_tile(tasks, n_tasks_p, tile_start, tl)) {
        if (threadIdx.x == 0) tile_left[blockIdx.x] = 0;
        return;
    }
    const SahTask T = tasks[tl.t];
    const int* src = T.buf ? idx1 : idx0;
    int cnt = 0;
    for (int j = tl.j0 + threadIdx.x; j < tl.j1; j += blockDim.x) {
        const int i = src[j];
        cnt += sah_goes_left(T, j, tlo[i], thi[i], nb);
    }
    __shared__ int red;
    if (threadIdx.x == 0) red = 0;
    __syncthreads();
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) atomicAdd(&red, cnt);
    __syncthreads();
    if (threadIdx.x == 0) tile_left[blockIdx.x] = red;
}

// stable partition of each range into the other index buffer; tile_off = exclusive scan of tile_left over the grid
__global__ void __launch_bounds__(256) k_sah_scatter(const SahTask* tasks, const int* n_tasks_p, const int* tile_start, int* idx0,
                                                     int* idx1, const float4* tlo, const float4* thi, int nb, const int* tile_off) {
    constexpr int PER = SAH_TILE / 256;
    SahTile tl;
    if (!sah_tile(tasks, n_tasks_p, tile_start, tl)) return;
    const SahTask T = tasks[tl.t];
    const int* src = T.buf ? idx1 : idx0;
    int* dst = T.buf ? idx0 : idx1;
    const int j0 = tl.j0 + threadIdx.x * PER;
    unsigned mask = 0;
    int vals[PER];
    for (int k = 0; k < PER; ++k) {
        const int j = j0 + k;
        vals[k] = j < tl.j1 ? src[j] : 0;
        if (j < tl.j1 && sah_goes_left(T, j, tlo[vals[k]], thi[vals[k]], nb)) mask |= 1u << k;
    }
    using Scan = cub::BlockScan<int, 256>;
    __shared__ typename Scan::TempStorage ts;
    int excl;
    Scan(ts).ExclusiveSum(__popc(mask), excl);
    int l = tile_off[blockIdx.x] - tile_off[tile_start[tl.t]] + excl;  // left primitives of the range before j0
    int r = (min(j0, tl.j1) - T.b) - l;
    for (int k = 0; k < PER; ++k) {
        const int j = j0 + k;
        if (j >= tl.j1) break;
        if (mask >> k & 1) dst[T.b + l++] = vals[k];
        else dst[T.mid + r++] = vals[k];
    }
}

// ---- ranges of at most SAH_T primitives: one CTA builds the whole subtree ----------------------------------------------

struct SahItem {
    int parent;
    unsigned short b, e;        // positions in the task's range
    unsigned short level, lanc; // relative to the task
};

// dynamic shared memory of k_sah_small
inline size_t sah_small_smem(int nb) {
    return size_t(SAH_T) * (6 * 4 + 2 * 2 + sizeof(SahItem)) + size_t(3) * nb * SAH_BIN_WORDS * 4;
}

__global__ void __launch_bounds__(SAH_SMALL_THREADS) k_sah_small(const SahTask* tasks, const int* idx0, const int* idx1,
                                                                 const float4* tlo, const float4* thi, SahParams p, SahTmp tmp,
                                                                 int* order) {
    constexpr int NT = SAH_SMALL_THREADS;
    extern __shared__ __align__(16) unsigned char smem[];
    float* s_box = reinterpret_cast<float*>(smem);  // [6][SAH_T]: lo xyz, hi xyz by local primitive
    SahItem* s_stack = reinterpret_cast<SahItem*>(s_box + 6 * SAH_T);
    unsigned short* s_perm = reinterpret_cast<unsigned short*>(s_stack + SAH_T);  // position -> local primitive
    unsigned short* s_tmp = s_perm + SAH_T;
    unsigned* s_bins = reinterpret_cast<unsigned*>(s_tmp + SAH_T);  // [3][nb][SAH_BIN_WORDS]
    __shared__ unsigned s_red[12];
    __shared__ SahItem s_cur;
    __shared__ int s_sp, s_mid, s_axis, s_split;
    __shared__ float s_cmin, s_scale;
    using Scan = cub::BlockScan<int, NT>;
    __shared__ typename Scan::TempStorage s_scan;

    const SahTask T = tasks[blockIdx.x];
    const int n = T.e - T.b, nb = p.n_bins, tid = threadIdx.x;
    const int* src = T.buf ? idx1 : idx0;
    for (int j = tid; j < n; j += NT) {
        const int i = src[T.b + j];
        const float4 l = tlo[i], h = thi[i];
        s_box[0 * SAH_T + j] = l.x; s_box[1 * SAH_T + j] = l.y; s_box[2 * SAH_T + j] = l.z;
        s_box[3 * SAH_T + j] = h.x; s_box[4 * SAH_T + j] = h.y; s_box[5 * SAH_T + j] = h.z;
        s_perm[j] = (unsigned short)j;
    }
    if (tid == 0) {
        s_stack[0] = SahItem{T.parent, 0, (unsigned short)n, 0, 0};
        s_sp = 1;
    }
    for (;;) {
        __syncthreads();
        if (tid < 12) s_red[tid] = 0;
        if (tid == 0) s_cur = s_sp ? s_stack[--s_sp] : SahItem{0, 0, 0, 0, 0};
        __syncthreads();
        const SahItem it = s_cur;
        const int b = it.b, e = it.e, m = e - b;
        if (m == 0) break;
        unsigned acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int j = b + tid; j < e; j += NT) {
            const int q = s_perm[j];
            sah_acc_prim(acc, make_float4(s_box[q], s_box[SAH_T + q], s_box[2 * SAH_T + q], 0.f),
                         make_float4(s_box[3 * SAH_T + q], s_box[4 * SAH_T + q], s_box[5 * SAH_T + q], 0.f));
        }
        for (int k = 0; k < 12; ++k) {
            const unsigned v = __reduce_max_sync(0xffffffffu, acc[k]);
            if ((tid & 31) == 0) atomicMax(&s_red[k], v);
        }
        __syncthreads();
        float lo[3], hi[3], clo[3], chi[3], scale[3];
        sah_decode(s_red, lo, hi, clo, chi);
        bool on[3];
        for (int a = 0; a < 3; ++a) {
            on[a] = m >= 2 && chi[a] > clo[a];
            scale[a] = on[a] ? float(nb) / (chi[a] - clo[a]) : 0.f;
        }
        if (m >= 2) {
            for (int k = tid; k < 3 * nb * SAH_BIN_WORDS; k += NT) s_bins[k] = 0;
            __syncthreads();
            for (int j = b + tid; j < e; j += NT) {
                const int q = s_perm[j];
                for (int a = 0; a < 3; ++a) {
                    if (!on[a]) continue;
                    const float c = 0.5f * s_box[a * SAH_T + q] + 0.5f * s_box[(3 + a) * SAH_T + q];
                    unsigned* w = s_bins + (a * nb + sah_bin(c, clo[a], scale[a], nb)) * SAH_BIN_WORDS;
                    for (int d = 0; d < 3; ++d) {
                        atomicMax(&w[d], ~sah_key(s_box[d * SAH_T + q]));
                        atomicMax(&w[3 + d], sah_key(s_box[(3 + d) * SAH_T + q]));
                    }
                    atomicAdd(&w[6], 1u);
                }
            }
            __syncthreads();
        }
        if (tid < 32) {
            double cost = INFINITY;
            int split = -1;
            if (tid < 3 && on[tid]) sah_sweep(s_bins + tid * nb * SAH_BIN_WORDS, nb, cost, split);
            const double c1 = __shfl_sync(0xffffffffu, cost, 1), c2 = __shfl_sync(0xffffffffu, cost, 2);
            const int s1 = __shfl_sync(0xffffffffu, split, 1), s2 = __shfl_sync(0xffffffffu, split, 2);
            if (tid == 0) {
                int axis = -1;
                double best = INFINITY;
                const double cs[3] = {cost, c1, c2};
                const int ss[3] = {split, s1, s2};
                for (int a = 0; a < 3; ++a)
                    if (cs[a] < best) { best = cs[a]; axis = a; split = ss[a]; }
                if (sah_leaf(m, it.parent < 0, axis, best, sah_half_area(lo, hi), p)) {
                    sah_link(tmp, it.parent, PTB_BVH_LEAF_REF(T.b + b, m), lo, hi);  // positions ascend in caller index
                    s_mid = -1;
                } else {
                    int left = m / 2;
                    if (axis >= 0) {
                        left = 0;
                        for (int k = 0; k < split; ++k) left += (int)s_bins[(axis * nb + k) * SAH_BIN_WORDS + 6];
                        s_cmin = clo[axis];
                        s_scale = scale[axis];
                    }
                    const int mid = b + left, id = T.b + mid - 1;
                    sah_node(tmp, id, T.b + b, T.b + e, T.level + it.level, T.lanc + it.lanc);
                    sah_link(tmp, it.parent, id, lo, hi);
                    s_mid = mid; s_axis = axis; s_split = split;
                    const unsigned short lv = (unsigned short)(it.level + 1);
                    s_stack[s_sp++] = SahItem{2 * id + 1, (unsigned short)mid, (unsigned short)e, lv, it.lanc};
                    s_stack[s_sp++] = SahItem{2 * id, (unsigned short)b, (unsigned short)mid, lv, (unsigned short)(it.lanc + 1)};
                }
            }
        }
        __syncthreads();
        const int mid = s_mid;
        if (mid < 0) continue;
        // stable partition of [b, e): each thread takes a contiguous chunk
        const int axis = s_axis, split = s_split;
        const float cmin = s_cmin, sc = s_scale;
        const int chunk = (m + NT - 1) / NT;
        const int j0 = b + min(tid * chunk, m), j1 = b + min((tid + 1) * chunk, m);
        unsigned mask = 0;
        for (int j = j0; j < j1; ++j) {
            const int q = s_perm[j];
            bool left;
            if (axis < 0) left = j - b < m / 2;
            else left = sah_bin(0.5f * s_box[axis * SAH_T + q] + 0.5f * s_box[(3 + axis) * SAH_T + q], cmin, sc, nb) < split;
            if (left) mask |= 1u << (j - j0);
        }
        int excl;
        Scan(s_scan).ExclusiveSum(__popc(mask), excl);
        int l = b + excl, r = mid + (j0 - b - excl);
        for (int j = j0; j < j1; ++j) {
            const unsigned short q = s_perm[j];
            if (mask >> (j - j0) & 1) s_tmp[l++] = q; else s_tmp[r++] = q;
        }
        __syncthreads();
        for (int j = b + tid; j < e; j += NT) s_perm[j] = s_tmp[j];
    }
    for (int j = tid; j < n; j += NT) order[T.b + j] = src[T.b + s_perm[j]];
}

// ---- renumbering: breadth-first prefix, then depth-first subtrees (bvh_build.cpp build_bvh) ------------------------------
// Breadth-first order is (level, b) order: a level's nodes are disjoint ranges, queued left to right.  When the prefix stops,
// the host queue holds the rest of the last level it reached, then the children of that level's nodes it took: the leftmost
// nodes of the next level.  In (level, b) order that is one run of positions [want, qend).  Inside the subtree of a queued
// root R, node t sits at base(R) + (used ids in [b_R, b_t)) + lanc_t - lanc_R in depth-first pre-order, child0 first: the ids
// below b_t are the nodes left of t and the ancestors that hold t on their child1 side, and lanc counts the others.

__global__ void __launch_bounds__(256) k_sah_keys(const int* used, const int4* info, int n_slots, unsigned long long* keys, int* vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_slots) return;
    keys[i] = used[i] ? ((unsigned long long)(unsigned)info[i].z << 32) | (unsigned)info[i].x : ~0ull;
    vals[i] = i;
}

PTD_FI int sah_lower_bound(const unsigned long long* a, int n, unsigned long long v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (a[m] < v) lo = m + 1; else hi = m;
    }
    return lo;
}

// meta: n_nodes, want (the breadth-first prefix), end of the prefix's last level, qend; base[q]: first position of queued root q
__global__ void __launch_bounds__(1024) k_sah_queue(const unsigned long long* skeys, const int* svals, const int* P, int n, int smem_nodes,
                                                    const int4* info, const int2* child, int* base, int* meta) {
    using Scan = cub::BlockScan<int, 1024>;
    __shared__ typename Scan::TempStorage ts;
    __shared__ int s_m, carry;
    const int n_nodes = P[n - 1];
    const int want = min(max(smem_nodes, 1), n_nodes);
    const unsigned long long lam = skeys[want - 1] >> 32;
    const int lvl_lo = sah_lower_bound(skeys, n_nodes, lam << 32), lvl_hi = sah_lower_bound(skeys, n_nodes, (lam + 1) << 32);
    if (threadIdx.x == 0) { s_m = 0; carry = 0; }
    __syncthreads();
    int m = 0;
    for (int s = lvl_lo + threadIdx.x; s < want; s += blockDim.x) {
        const int2 c = child[svals[s]];
        m += (c.x >= 0) + (c.y >= 0);
    }
    m = __reduce_add_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_m, m);
    __syncthreads();
    const int qend = lvl_hi + s_m;
    for (int s0 = want; s0 < qend; s0 += 1024) {
        const int s = s0 + threadIdx.x;
        int size = 0;
        if (s < qend) {
            const int4 in = info[svals[s]];
            size = P[in.y - 1] - P[in.x];
        }
        int excl, total;
        Scan(ts).ExclusiveSum(size, excl, total);
        if (s < qend) base[s - want] = want + carry + excl;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) { meta[0] = n_nodes; meta[1] = want; meta[2] = lvl_hi; meta[3] = qend; }
}

// last position r in [lo, hi) whose range starts at or before bt
PTD_FI int sah_last_le(const unsigned long long* skeys, int lo, int hi, unsigned bt) {
    while (hi - lo > 1) {
        const int m = (lo + hi) >> 1;
        if ((unsigned)(skeys[m] & 0xffffffffu) <= bt) lo = m; else hi = m;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_sah_newid(const unsigned long long* skeys, const int* svals, const int* P, const int4* info,
                                                   const int* base, const int* meta, int* new_of) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_nodes = meta[0], want = meta[1], g1_end = meta[2], qend = meta[3];
    if (s >= n_nodes) return;
    const int t = svals[s];
    if (s < want) { new_of[t] = s; return; }
    const unsigned bt = (unsigned)(skeys[s] & 0xffffffffu);
    // queued roots: [want, g1_end) the rest of the last prefix level, [g1_end, qend) next-level nodes left of all of them
    const bool in_g1 = g1_end > want && (unsigned)(skeys[want] & 0xffffffffu) <= bt;
    const int r = in_g1 ? sah_last_le(skeys, want, g1_end, bt) : sah_last_le(skeys, g1_end, qend, bt);
    const int4 ir = info[svals[r]], it = info[t];
    new_of[t] = base[r - want] + (P[it.x] - P[ir.x]) + (it.w - ir.w);
}

// the ptb_bvh_node records: children renumbered, boxes padded and encoded as the host and k_lbvh_finish do
__global__ void __launch_bounds__(256) k_sah_emit(const int* svals, const int* meta, const int* new_of, const int2* child,
                                                  const float4* box, float pad_rel, const int* scene_bounds, float4* nodes) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= meta[0]) return;
    const int t = svals[s];
    const float dx = ordered_to_float(scene_bounds[3]) - ordered_to_float(scene_bounds[0]);
    const float dy = ordered_to_float(scene_bounds[4]) - ordered_to_float(scene_bounds[1]);
    const float dz = ordered_to_float(scene_bounds[5]) - ordered_to_float(scene_bounds[2]);
    const float pad = pad_rel * sqrtf(dx * dx + dy * dy + dz * dz);
    auto ce = [pad](float lo, float hi, float& cc, float& ee) {
        lo -= pad; hi += pad;
        cc = 0.5f * lo + 0.5f * hi;
        const float h = 0.5f * hi - 0.5f * lo;
        ee = h + 2.4e-7f * (fabsf(cc) + h);
    };
    const int2 c = child[t];
    const int r0 = c.x >= 0 ? new_of[c.x] : c.x, r1 = c.y >= 0 ? new_of[c.y] : c.y;
    const float4 l0 = box[4 * (size_t)t], h0 = box[4 * (size_t)t + 1], l1 = box[4 * (size_t)t + 2], h1 = box[4 * (size_t)t + 3];
    float4 o0, o1, o2, o3;
    ce(l0.x, h0.x, o0.x, o1.x); ce(l0.y, h0.y, o0.y, o1.y); ce(l0.z, h0.z, o0.z, o1.z);
    ce(l1.x, h1.x, o2.x, o3.x); ce(l1.y, h1.y, o2.y, o3.y); ce(l1.z, h1.z, o2.z, o3.z);
    o0.w = __int_as_float(r0); o1.w = __int_as_float(r1); o2.w = 0.f; o3.w = 0.f;
    float4* nd = nodes + 4 * (size_t)new_of[t];
    nd[0] = o0; nd[1] = o1; nd[2] = o2; nd[3] = o3;
}

// precomputed-edge triangles in leaf order (as k_lbvh_finish)
__global__ void __launch_bounds__(256) k_sah_tris(const ptb_triangle* tris, const int* order, int n, float4* otris) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int tri = order[i];
    const float4* p = reinterpret_cast<const float4*>(tris + tri);
    const float4 p1 = p[0], p2 = p[1], p3 = p[2];
    const int quad = reinterpret_cast<const int*>(tris + tri)[12];
    otris[3 * (size_t)i + 0] = make_float4(p1.x, p1.y, p1.z, __int_as_float(tri));
    otris[3 * (size_t)i + 1] = make_float4(p2.x - p1.x, p2.y - p1.y, p2.z - p1.z, __int_as_float(quad));  // GenerateColors.cl:92
    otris[3 * (size_t)i + 2] = make_float4(p3.x - p1.x, p3.y - p1.y, p3.z - p1.z, 0.f);                   // GenerateColors.cl:93
}

__global__ void k_sah_root(int n, SahTask* large, SahTask* small, int* counts) {
    SahTask r{};
    r.b = 0; r.e = n; r.parent = -1; r.level = 1;
    if (n > SAH_T) { large[0] = r; counts[0] = 1; counts[1] = 0; }
    else { small[0] = r; counts[0] = 0; counts[1] = 1; }
}

__global__ void __launch_bounds__(256) k_sah_iota(int* idx, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = i;
}

// The SAH tree of n caller-order records on the device (n >= 2): outputs as build_lbvh_device, plus the node count and the
// breadth-first prefix.  The `readback` bytes come back in the last synchronisation.
static int build_sah_device(cudaStream_t st, const ptb_triangle* d_tris, int n, const ptb_bvh_params& bp, float4** d_nodes_out,
                            float4** d_otris_out, int** d_order_out, int* n_nodes_out, int* depth_out, int* bfs_out,
                            const void* d_readback, void* h_readback, size_t readback) {
    int rc = PTB_OK;
    SahParams p;
    p.max_leaf = min(max(bp.max_leaf, 1), PTB_BVH_MAX_LEAF);
    p.n_bins = min(max(bp.n_bins, 2), 256);
    p.k_traverse = bp.traverse_cost > 0.0f ? double(bp.traverse_cost) : 1.2;
    const int nb = p.n_bins;
    const int cap_level = n / (SAH_T + 1) + 1;  // disjoint ranges of more than SAH_T
    const int cap_tiles = n / SAH_TILE + 1 + cap_level;
    float4 *tlo = nullptr, *thi = nullptr, *nodes = nullptr, *otris = nullptr;
    int *misc = nullptr, *idx0 = nullptr, *idx1 = nullptr, *order = nullptr, *tile_start = nullptr, *tile_left = nullptr,
        *tile_off = nullptr, *P = nullptr, *vals = nullptr, *svals = nullptr, *new_of = nullptr, *base = nullptr;
    SahTask *lev[2] = {nullptr, nullptr}, *small = nullptr;
    unsigned *tb = nullptr, *bins = nullptr;
    unsigned long long *keys = nullptr, *skeys = nullptr;
    SahTmp tmp{};
    char* arena = nullptr;
    unsigned char* temp = nullptr;
    size_t temp_bytes = 0, tb_scan = 0, tb_p = 0, tb_sort = 0;
    int counts[2] = {n > SAH_T ? 1 : 0, n > SAH_T ? 0 : 1};  // large ranges of this level, small ranges so far
    int meta[4], depth = 0, cur = 0;
    const int grid_n = (n + 255) / 256, n_slots = n - 1;
    const size_t small_smem = sah_small_smem(nb);
    // one arena for the scratch arrays (two passes: measure, then carve); misc: [0, 6) scene bounds, 6 root id, 7 max level,
    // 8 next-level count, 9 small count, [10, 14) meta, 14 this level's count
    LBVH_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb_scan, tile_left, tile_off, cap_tiles, st));
    LBVH_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb_p, tmp.used, P, n, st));
    LBVH_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, keys, skeys, vals, svals, n_slots, 0, 64, st));
    temp_bytes = max(tb_scan, max(tb_p, tb_sort));
    for (int pass = 0; pass < 2; ++pass) {
        size_t off = 0;
        auto carve = [&](auto** q, size_t bytes) {
            *q = reinterpret_cast<std::remove_reference_t<decltype(**q)>*>(arena + off);
            off += (bytes + 255) & ~size_t(255);
        };
        carve(&tlo, sizeof(float4) * (size_t)n); carve(&thi, sizeof(float4) * (size_t)n);
        carve(&misc, 4 * 16);
        carve(&idx0, 4 * (size_t)n); carve(&idx1, 4 * (size_t)n);
        carve(&lev[0], sizeof(SahTask) * (size_t)cap_level); carve(&lev[1], sizeof(SahTask) * (size_t)cap_level);
        carve(&small, sizeof(SahTask) * (size_t)n);
        carve(&tb, 48 * (size_t)cap_level);
        carve(&tile_start, 4 * (size_t)(cap_level + 1));
        carve(&tile_left, 4 * (size_t)cap_tiles); carve(&tile_off, 4 * (size_t)cap_tiles);
        carve(&tmp.child, sizeof(int2) * (size_t)n_slots);
        carve(&tmp.box, 4 * sizeof(float4) * (size_t)n_slots);
        carve(&tmp.info, sizeof(int4) * (size_t)n_slots);
        carve(&tmp.used, 4 * (size_t)n);
        carve(&P, 4 * (size_t)n);
        carve(&keys, 8 * (size_t)n_slots); carve(&skeys, 8 * (size_t)n_slots);
        carve(&vals, 4 * (size_t)n_slots); carve(&svals, 4 * (size_t)n_slots);
        carve(&new_of, 4 * (size_t)n_slots); carve(&base, 4 * (size_t)n_slots);
        carve(&temp, temp_bytes);
        if (pass == 0) LBVH_TRY(cudaMalloc((void**)&arena, off));
    }
    LBVH_TRY(cudaMalloc((void**)&order, 4 * (size_t)n));
    LBVH_TRY(cudaFuncSetAttribute(k_sah_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem));
    tmp.root_id = misc + 6;
    tmp.max_level = misc + 7;
    LBVH_TRY(cudaMemsetAsync(misc, 0, 4 * 16, st));
    LBVH_TRY(cudaMemsetAsync(tmp.used, 0, 4 * (size_t)n, st));
    k_lbvh_init<<<1, 32, 0, st>>>(misc);
    k_lbvh_tri_bounds<<<grid_n, 256, 0, st>>>(d_tris, n, tlo, thi, misc);
    k_sah_iota<<<grid_n, 256, 0, st>>>(idx0, n);
    k_sah_root<<<1, 1, 0, st>>>(n, lev[0], small, misc + 8);
    LBVH_TRY(cudaGetLastError());
    for (int bins_cap = 0; counts[0] > 0; cur ^= 1) {
        const int nt = counts[0];
        const size_t bin_words = (size_t)nt * 3 * nb * SAH_BIN_WORDS;
        if (nt > bins_cap) {
            if (bins) cudaFree(bins);
            bins = nullptr;
            LBVH_TRY(cudaMalloc((void**)&bins, 4 * bin_words));
            bins_cap = nt;
        }
        const int grid = n / SAH_TILE + 1 + nt;
        int* n_tasks = misc + 8;  // this level's count, then the next level's
        LBVH_TRY(cudaMemsetAsync(tb, 0, 48 * (size_t)nt, st));
        LBVH_TRY(cudaMemsetAsync(bins, 0, 4 * bin_words, st));
        k_sah_plan<<<1, 1024, 0, st>>>(lev[cur], n_tasks, tile_start);
        k_sah_bounds<<<grid, 256, 0, st>>>(lev[cur], n_tasks, tile_start, idx0, idx1, tlo, thi, tb);
        k_sah_bin<<<grid, 256, 0, st>>>(lev[cur], n_tasks, tile_start, idx0, idx1, tlo, thi, tb, nb, bins);
        LBVH_TRY(cudaMemcpyAsync(misc + 14, n_tasks, 4, cudaMemcpyDeviceToDevice, st));  // keep this level's count
        LBVH_TRY(cudaMemsetAsync(n_tasks, 0, 4, st));
        k_sah_decide<<<(nt * 32 + 127) / 128, 128, 0, st>>>(lev[cur], misc + 14, tb, bins, p, tmp, lev[cur ^ 1], n_tasks, small, misc + 9);
        k_sah_count<<<grid, 256, 0, st>>>(lev[cur], misc + 14, tile_start, idx0, idx1, tlo, thi, nb, tile_left);
        LBVH_TRY(cub::DeviceScan::ExclusiveSum(temp, tb_scan, tile_left, tile_off, grid, st));
        k_sah_scatter<<<grid, 256, 0, st>>>(lev[cur], misc + 14, tile_start, idx0, idx1, tlo, thi, nb, tile_off);
        LBVH_TRY(cudaGetLastError());
        LBVH_TRY(cudaMemcpyAsync(counts, misc + 8, 8, cudaMemcpyDeviceToHost, st));
        LBVH_TRY(cudaStreamSynchronize(st));
    }
    k_sah_small<<<counts[1], SAH_SMALL_THREADS, small_smem, st>>>(small, idx0, idx1, tlo, thi, p, tmp, order);
    k_sah_keys<<<(n_slots + 255) / 256, 256, 0, st>>>(tmp.used, tmp.info, n_slots, keys, vals);
    LBVH_TRY(cudaGetLastError());
    LBVH_TRY(cub::DeviceScan::ExclusiveSum(temp, tb_p, tmp.used, P, n, st));
    LBVH_TRY(cub::DeviceRadixSort::SortPairs(temp, tb_sort, keys, skeys, vals, svals, n_slots, 0, 64, st));
    k_sah_queue<<<1, 1024, 0, st>>>(skeys, svals, P, n, bp.smem_nodes, tmp.info, tmp.child, base, misc + 10);
    LBVH_TRY(cudaGetLastError());
    LBVH_TRY(cudaMemcpyAsync(meta, misc + 10, 16, cudaMemcpyDeviceToHost, st));
    LBVH_TRY(cudaMemcpyAsync(&depth, tmp.max_level, 4, cudaMemcpyDeviceToHost, st));
    LBVH_TRY(cudaStreamSynchronize(st));
    LBVH_TRY(cudaMalloc((void**)&nodes, 64 * (size_t)meta[0]));
    LBVH_TRY(cudaMalloc((void**)&otris, 48 * (size_t)n));
    k_sah_newid<<<(meta[0] + 255) / 256, 256, 0, st>>>(skeys, svals, P, tmp.info, base, misc + 10, new_of);
    k_sah_emit<<<(meta[0] + 255) / 256, 256, 0, st>>>(svals, misc + 10, new_of, tmp.child, tmp.box, bp.pad_rel, misc, nodes);
    k_sah_tris<<<grid_n, 256, 0, st>>>(d_tris, order, n, otris);
    LBVH_TRY(cudaGetLastError());
    if (readback) LBVH_TRY(cudaMemcpyAsync(h_readback, d_readback, readback, cudaMemcpyDeviceToHost, st));
    LBVH_TRY(cudaStreamSynchronize(st));
    *d_nodes_out = nodes; *d_otris_out = otris; *d_order_out = order;
    *n_nodes_out = meta[0]; *depth_out = depth; *bfs_out = meta[1];
    nodes = nullptr; otris = nullptr; order = nullptr;
cleanup:
    for (void* q : {(void*)arena, (void*)order, (void*)bins, (void*)nodes, (void*)otris})
        if (q) cudaFree(q);
    return rc;
}

}  // namespace ptd
