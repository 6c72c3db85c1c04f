// bvh_build.cpp -- deterministic host BVH builder (BUILD-DEFINED: the reference
// has no acceleration structure; every ray loops over NUM_TRIANGLES,
// test/ClKernels/GenerateColors.cl:137-154).
//
// Output format (include/SharedHeader.h): binary 64-byte nodes (and, for small scenes, the same tree
// collapsed to 128-byte 4-wide nodes) holding their children's padded boxes as centre/half-extent,
// 48-byte precomputed-edge triangles in leaf order.
// The tree must be EQUIVALENT to the brute-force loop: traversal may only skip
// triangles the Moller-Trumbore test would reject, so every stored box is the
// exact fp32 bound of its triangles grown by an absolute pad (pad_rel x scene
// diagonal) that dominates the rounding of both the slab test and the
// triangle test (DESIGN.md "BVH equivalence").
//
// Algorithm: top-down binned SAH (n_bins centroid bins per axis, axes tried in
// x,y,z order, first strictly-lowest cost wins), leaf when count <= max_leaf and
// splitting does not pay; median split when no bin boundary separates the set.
// Triangles inside a leaf are kept in ascending caller index.  After the build
// the first `smem_nodes` nodes are renumbered breadth-first (one contiguous
// block that a CTA stages in shared memory with a single bulk copy); the
// remaining subtrees follow depth-first.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>

#include "host_internal.h"

namespace ptb {
namespace {

struct Prim {
    float lo[3], hi[3], c[3];
    int32_t idx;
};

struct Box {
    float lo[3], hi[3];
    void reset() {
        for (int a = 0; a < 3; ++a) { lo[a] = INFINITY; hi[a] = -INFINITY; }
    }
    void grow(const float* l, const float* h) {
        for (int a = 0; a < 3; ++a) { lo[a] = std::min(lo[a], l[a]); hi[a] = std::max(hi[a], h[a]); }
    }
    double half_area() const {
        const double dx = double(hi[0]) - lo[0], dy = double(hi[1]) - lo[1], dz = double(hi[2]) - lo[2];
        return dx * dy + dy * dz + dz * dx;
    }
};

struct TmpNode {
    int32_t child[2];
    Box box[2];
};

struct Builder {
    std::vector<Prim> prims;
    std::vector<TmpNode> nodes;
    std::vector<int32_t> order;  // leaf order -> caller index
    int max_leaf, n_bins;
    static constexpr double kIntersect = 1.0;
    double kTraverse = 1.2;  // ptb_bvh_params.traverse_cost

    // returns child reference; fills the exact bounds of [b, e)
    int32_t build(int b, int e, bool force_split, Box* bounds) {
        const int n = e - b;
        Box bb, cb;
        bb.reset(); cb.reset();
        for (int i = b; i < e; ++i) { bb.grow(prims[i].lo, prims[i].hi); cb.grow(prims[i].c, prims[i].c); }
        *bounds = bb;

        int best_axis = -1, best_split = -1;
        double best_cost = INFINITY;
        if (n >= 2) {
            std::vector<Box> bin_box(n_bins);
            std::vector<int> bin_cnt(n_bins);
            std::vector<double> right_area(n_bins);
            std::vector<int> right_cnt(n_bins);
            for (int axis = 0; axis < 3; ++axis) {
                const float cmin = cb.lo[axis], cmax = cb.hi[axis];
                if (!(cmax > cmin)) continue;
                const float scale = float(n_bins) / (cmax - cmin);
                for (int k = 0; k < n_bins; ++k) { bin_box[k].reset(); bin_cnt[k] = 0; }
                for (int i = b; i < e; ++i) {
                    const int k = bin_of(prims[i].c[axis], cmin, scale);
                    bin_box[k].grow(prims[i].lo, prims[i].hi);
                    bin_cnt[k]++;
                }
                Box acc; acc.reset(); int cnt = 0;
                for (int k = n_bins - 1; k >= 1; --k) {
                    if (bin_cnt[k]) acc.grow(bin_box[k].lo, bin_box[k].hi);
                    cnt += bin_cnt[k];
                    right_area[k] = cnt ? acc.half_area() : 0.0;
                    right_cnt[k] = cnt;
                }
                acc.reset(); cnt = 0;
                for (int k = 1; k < n_bins; ++k) {  // split between bin k-1 and k
                    if (bin_cnt[k - 1]) acc.grow(bin_box[k - 1].lo, bin_box[k - 1].hi);
                    cnt += bin_cnt[k - 1];
                    if (cnt == 0 || right_cnt[k] == 0) continue;
                    const double cost = acc.half_area() * cnt + right_area[k] * right_cnt[k];
                    if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = k; }
                }
            }
        }

        const double parent_area = bb.half_area();
        const double split_cost = (best_axis >= 0 && parent_area > 0.0)
                                      ? kTraverse + kIntersect * best_cost / parent_area
                                      : (best_axis >= 0 ? kTraverse : INFINITY);
        const bool can_leaf = n <= max_leaf && !force_split;
        if (n == 1 || (can_leaf && double(n) * kIntersect <= split_cost)) return make_leaf(b, e);

        int mid;
        if (best_axis >= 0) {
            const float cmin = cb.lo[best_axis];
            const float scale = float(n_bins) / (cb.hi[best_axis] - cmin);
            mid = b;
            for (int i = b; i < e; ++i)  // in-place, order-preserving on the left side
                if (bin_of(prims[i].c[best_axis], cmin, scale) < best_split) std::swap(prims[i], prims[mid++]);
        } else {
            // no separating bin boundary: order by caller index and cut in half
            std::sort(prims.begin() + b, prims.begin() + e, [](const Prim& x, const Prim& y) { return x.idx < y.idx; });
            mid = b + n / 2;
        }
        const int32_t me = int32_t(nodes.size());
        nodes.emplace_back();
        Box lb, rb;
        const int32_t l = build(b, mid, false, &lb);
        const int32_t r = build(mid, e, false, &rb);
        nodes[me].child[0] = l; nodes[me].child[1] = r;
        nodes[me].box[0] = lb; nodes[me].box[1] = rb;
        return me;
    }

    int bin_of(float c, float cmin, float scale) const {
        int k = int((c - cmin) * scale);
        return k < 0 ? 0 : (k >= n_bins ? n_bins - 1 : k);
    }

    int32_t make_leaf(int b, int e) {
        std::sort(prims.begin() + b, prims.begin() + e, [](const Prim& x, const Prim& y) { return x.idx < y.idx; });
        const int first = int(order.size());
        for (int i = b; i < e; ++i) order.push_back(prims[i].idx);
        return PTB_BVH_LEAF_REF(first, e - b);
    }
};

// [lo, hi] -> centre / half-extent, widened by two ulps so that [c - e, c + e] still contains [lo, hi]
void centre_extent(float lo, float hi, float* c, float* e) {
    *c = 0.5f * lo + 0.5f * hi;
    const float h = 0.5f * hi - 0.5f * lo;
    *e = h + 2.4e-7f * (std::fabs(*c) + h);
}

void edge_tri(const ptb_triangle& t, int32_t index, ptb_bvh_tri* o) {
    const float* p1 = &t.p1.x;
    const float* p2 = &t.p2.x;
    const float* p3 = &t.p3.x;
    for (int a = 0; a < 3; ++a) {
        o->p1[a] = p1[a];
        o->e1[a] = p2[a] - p1[a];  // GenerateColors.cl:92
        o->e2[a] = p3[a] - p1[a];  // GenerateColors.cl:93
    }
    o->index = index;
    o->quad = t.id;
    o->pad = 0;
}

}  // namespace

void make_edge_tris(const ptb_triangle* tris, int n_tris, std::vector<ptb_bvh_tri>* out) {
    out->resize(size_t(n_tris));
    for (int i = 0; i < n_tris; ++i) edge_tri(tris[i], i, &(*out)[i]);
}

int build_bvh(const ptb_triangle* tris, int n_tris, const ptb_bvh_params& params, BuiltBvh* out) {
    if (!tris || n_tris < 1 || !out) return fail(PTB_E_INVALID, "build_bvh: need at least one triangle");
    if (n_tris >= (1 << 28)) return fail(PTB_E_INVALID, "build_bvh: too many triangles for the leaf encoding");
    if (!(params.pad_rel > 0.0f) || std::isinf(params.pad_rel))
        return fail(PTB_E_INVALID, "build_bvh: pad_rel must be a finite number > 0, got %g (without a pad, rounding in the box "
                    "and triangle tests loses hits)", double(params.pad_rel));
    Builder B;
    B.max_leaf = std::min(std::max(params.max_leaf, 1), PTB_BVH_MAX_LEAF);
    B.n_bins = std::min(std::max(params.n_bins, 2), 256);
    if (params.traverse_cost > 0.0f) B.kTraverse = params.traverse_cost;
    B.prims.resize(size_t(n_tris));
    Box scene; scene.reset();
    for (int i = 0; i < n_tris; ++i) {
        Prim& p = B.prims[i];
        const float* v[3] = {&tris[i].p1.x, &tris[i].p2.x, &tris[i].p3.x};
        for (int a = 0; a < 3; ++a) {
            p.lo[a] = std::min(v[0][a], std::min(v[1][a], v[2][a]));
            p.hi[a] = std::max(v[0][a], std::max(v[1][a], v[2][a]));
            if (!(p.lo[a] == p.lo[a]) || !(p.hi[a] == p.hi[a]) || std::isinf(p.lo[a]) || std::isinf(p.hi[a]))
                return fail(PTB_E_INVALID, "build_bvh: triangle %d has a non-finite vertex", i);
            p.c[a] = 0.5f * p.lo[a] + 0.5f * p.hi[a];
        }
        p.idx = i;
        scene.grow(p.lo, p.hi);
    }
    B.nodes.reserve(size_t(n_tris));
    B.order.reserve(size_t(n_tris));

    if (n_tris == 1) {
        // a root must be an internal node: both binary children are the same one-triangle leaf
        TmpNode root;
        root.child[0] = root.child[1] = B.make_leaf(0, 1);
        root.box[0] = root.box[1] = scene;
        B.nodes.push_back(root);
    } else {
        Box bb;
        const int32_t r = B.build(0, n_tris, /*force_split=*/true, &bb);
        if (r != 0) return fail(PTB_E_INVALID, "build_bvh: internal error (root ref %d)", r);
    }

    // pad: absolute, relative to the scene diagonal
    const float dx = scene.hi[0] - scene.lo[0], dy = scene.hi[1] - scene.lo[1], dz = scene.hi[2] - scene.lo[2];
    const float diag = std::sqrt(dx * dx + dy * dy + dz * dz);
    const float pad = params.pad_rel * diag;

    // renumber: breadth-first prefix, then depth-first subtrees
    const int n_nodes = int(B.nodes.size());
    const int want_bfs = std::min(std::max(params.smem_nodes, 1), n_nodes);
    std::vector<int32_t> new_of(size_t(n_nodes), -1);
    std::vector<int32_t> old_of;
    old_of.reserve(size_t(n_nodes));
    std::deque<int32_t> queue{0};
    while (!queue.empty() && int(old_of.size()) < want_bfs) {
        const int32_t o = queue.front();
        queue.pop_front();
        new_of[o] = int32_t(old_of.size());
        old_of.push_back(o);
        for (int c = 0; c < 2; ++c)
            if (B.nodes[o].child[c] >= 0) queue.push_back(B.nodes[o].child[c]);
    }
    const int bfs_count = int(old_of.size());
    std::vector<int32_t> stack;
    for (int32_t root : queue) {
        stack.push_back(root);
        while (!stack.empty()) {
            const int32_t o = stack.back();
            stack.pop_back();
            new_of[o] = int32_t(old_of.size());
            old_of.push_back(o);
            if (B.nodes[o].child[1] >= 0) stack.push_back(B.nodes[o].child[1]);
            if (B.nodes[o].child[0] >= 0) stack.push_back(B.nodes[o].child[0]);
        }
    }
    if (int(old_of.size()) != n_nodes) return fail(PTB_E_INVALID, "build_bvh: renumbering lost nodes");

    out->nodes.assign(size_t(n_nodes), ptb_bvh_node{});
    for (int ni = 0; ni < n_nodes; ++ni) {
        const TmpNode& t = B.nodes[old_of[ni]];
        ptb_bvh_node& d = out->nodes[ni];
        d.child0 = t.child[0] >= 0 ? new_of[t.child[0]] : t.child[0];
        d.child1 = t.child[1] >= 0 ? new_of[t.child[1]] : t.child[1];
        for (int a = 0; a < 3; ++a) {
            centre_extent(t.box[0].lo[a] - pad, t.box[0].hi[a] + pad, &d.c0[a], &d.e0[a]);
            centre_extent(t.box[1].lo[a] - pad, t.box[1].hi[a] + pad, &d.c1[a], &d.e1[a]);
        }
        d.pad0 = d.pad1 = 0;
    }
    // depth = longest chain of internal nodes (bounds the traversal stack)
    int depth = 1;
    {
        std::vector<std::pair<int32_t, int>> st{{0, 1}};
        while (!st.empty()) {
            auto [ni, dep] = st.back();
            st.pop_back();
            depth = std::max(depth, dep);
            if (out->nodes[ni].child0 >= 0) st.push_back({out->nodes[ni].child0, dep + 1});
            if (out->nodes[ni].child1 >= 0) st.push_back({out->nodes[ni].child1, dep + 1});
        }
    }
    out->depth = depth;
    out->smem_nodes = bfs_count;

    if (n_tris <= PTB_FLAT_MAX_TRIS) {  // tiny scenes also get the FLAT form: every leaf slot with its box and triangle mask
        std::vector<ptb_bvh_leafbox> flat;
        bool fits = true;
        // leaf order == depth-first order with slot 0 first
        std::vector<std::pair<int32_t, int>> st;
        if (n_tris > 1) st.push_back({0, 1});  // the one-triangle root repeats its leaf in both slots
        st.push_back({0, 0});
        while (!st.empty()) {
            const auto [ni, slot] = st.back();
            st.pop_back();
            const int32_t r = B.nodes[ni].child[slot];
            if (r >= 0) { st.push_back({r, 1}); st.push_back({r, 0}); continue; }
            if (int(flat.size()) >= PTB_FLAT_MAX_LEAVES) { fits = false; break; }
            const int first = PTB_BVH_LEAF_FIRST(r), count = PTB_BVH_LEAF_COUNT(r);
            const uint64_t m = ((uint64_t(1) << count) - 1) << first;
            ptb_bvh_leafbox lb;
            for (int a = 0; a < 3; ++a) centre_extent(B.nodes[ni].box[slot].lo[a] - pad, B.nodes[ni].box[slot].hi[a] + pad, &lb.c[a], &lb.e[a]);
            lb.mask_lo = uint32_t(m); lb.mask_hi = uint32_t(m >> 32);
            flat.push_back(lb);
        }
        if (fits) out->flat = flat;
    }

    if (n_tris <= 2048) {  // small scenes also get the 4-wide form (shared-memory-resident traversal)
        // collapse the binary tree into 4-wide nodes: start from a node's two children and keep replacing the
        // internal child with the largest box (ties: lowest slot) by its own two children, in place, until four
        // slots are used or only leaves remain.
        struct Wide {
            int32_t child[PTB_BVH_WIDTH];
            Box box[PTB_BVH_WIDTH];
            int n = 0;
        };
        std::vector<Wide> wide;
        wide.reserve(B.nodes.size() / 2 + 1);
        {
            struct Item { int32_t bin; int32_t wide_parent; int slot; };
            std::vector<Item> todo{{0, -1, 0}};
            while (!todo.empty()) {
                const Item it = todo.back();
                todo.pop_back();
                std::vector<std::pair<int32_t, Box>> slots;
                slots.push_back({B.nodes[it.bin].child[0], B.nodes[it.bin].box[0]});
                slots.push_back({B.nodes[it.bin].child[1], B.nodes[it.bin].box[1]});
                while (int(slots.size()) < PTB_BVH_WIDTH) {
                    int pick = -1;
                    double best = -1.0;
                    for (int k = 0; k < int(slots.size()); ++k)
                        if (slots[k].first >= 0 && slots[k].second.half_area() > best) { best = slots[k].second.half_area(); pick = k; }
                    if (pick < 0) break;
                    const TmpNode& t = B.nodes[slots[pick].first];
                    const std::pair<int32_t, Box> l{t.child[0], t.box[0]}, r{t.child[1], t.box[1]};
                    slots[pick] = l;
                    slots.insert(slots.begin() + pick + 1, r);
                }
                const int32_t me = int32_t(wide.size());
                wide.emplace_back();
                if (it.wide_parent >= 0) wide[it.wide_parent].child[it.slot] = me;
                wide[me].n = int(slots.size());
                for (int k = 0; k < PTB_BVH_WIDTH; ++k) {
                    if (k < int(slots.size())) {
                        wide[me].child[k] = slots[k].first;  // binary index for now (>= 0) or a leaf reference
                        wide[me].box[k] = slots[k].second;
                    } else {
                        wide[me].child[k] = PTB_BVH_EMPTY;
                    }
                }
                for (int k = int(slots.size()) - 1; k >= 0; --k)  // reverse push -> children are numbered in slot order
                    if (slots[k].first >= 0) todo.push_back({slots[k].first, me, k});
            }
        }

        // renumber: breadth-first prefix, then depth-first subtrees
        const int n_nodes = int(wide.size());
        const int want_bfs = std::min(std::max(params.smem_nodes, 1), n_nodes);
        std::vector<int32_t> new_of(size_t(n_nodes), -1);
        std::vector<int32_t> old_of;
        old_of.reserve(size_t(n_nodes));
        auto internal = [](int32_t ref) { return ref >= 0 && ref != PTB_BVH_EMPTY; };
        std::deque<int32_t> queue{0};
        while (!queue.empty() && int(old_of.size()) < want_bfs) {
            const int32_t o = queue.front();
            queue.pop_front();
            new_of[o] = int32_t(old_of.size());
            old_of.push_back(o);
            for (int c = 0; c < PTB_BVH_WIDTH; ++c)
                if (internal(wide[o].child[c])) queue.push_back(wide[o].child[c]);
        }
        const int bfs_count = int(old_of.size());
        std::vector<int32_t> stack;
        for (int32_t root : queue) {
            stack.push_back(root);
            while (!stack.empty()) {
                const int32_t o = stack.back();
                stack.pop_back();
                new_of[o] = int32_t(old_of.size());
                old_of.push_back(o);
                for (int c = PTB_BVH_WIDTH - 1; c >= 0; --c)
                    if (internal(wide[o].child[c])) stack.push_back(wide[o].child[c]);
            }
        }
        if (int(old_of.size()) != n_nodes) return fail(PTB_E_INVALID, "build_bvh: renumbering lost nodes");

        out->nodes4.assign(size_t(n_nodes), ptb_bvh_node4{});
        for (int ni = 0; ni < n_nodes; ++ni) {
            const Wide& t = wide[old_of[ni]];
            ptb_bvh_node4& d = out->nodes4[ni];
            float* cs[PTB_BVH_WIDTH] = {d.c0, d.c1, d.c2, d.c3};
            float* es[PTB_BVH_WIDTH] = {d.e0, d.e1, d.e2, d.e3};
            int32_t* refs[PTB_BVH_WIDTH] = {&d.child0, &d.child1, &d.child2, &d.child3};
            for (int k = 0; k < PTB_BVH_WIDTH; ++k) {
                *refs[k] = internal(t.child[k]) ? new_of[t.child[k]] : t.child[k];
                for (int a = 0; a < 3; ++a) {
                    if (t.child[k] == PTB_BVH_EMPTY) { cs[k][a] = 0.0f; es[k][a] = -1e30f; }
                    else centre_extent(t.box[k].lo[a] - pad, t.box[k].hi[a] + pad, &cs[k][a], &es[k][a]);
                }
            }
            d.pad0 = d.pad1 = d.pad2 = d.pad3 = 0;
        }
        // depth = longest chain of internal nodes (bounds the traversal stack: up to 3 deferred children per level)
        int depth = 1;
        {
            std::vector<std::pair<int32_t, int>> st{{0, 1}};
            while (!st.empty()) {
                auto [ni, dep] = st.back();
                st.pop_back();
                depth = std::max(depth, dep);
                const int32_t refs[PTB_BVH_WIDTH] = {out->nodes4[ni].child0, out->nodes4[ni].child1, out->nodes4[ni].child2, out->nodes4[ni].child3};
                for (int k = 0; k < PTB_BVH_WIDTH; ++k)
                    if (internal(refs[k])) st.push_back({refs[k], dep + 1});
            }
        }
        out->depth4 = depth;
        out->smem_nodes4 = bfs_count;
    }
    out->tri_order = B.order;
    out->tris.resize(B.order.size());
    for (size_t k = 0; k < B.order.size(); ++k) edge_tri(tris[B.order[k]], B.order[k], &out->tris[k]);
    for (int a = 0; a < 3; ++a) { out->scene_lo[a] = scene.lo[a]; out->scene_hi[a] = scene.hi[a]; }
    return PTB_OK;
}

}  // namespace ptb

extern "C" void ptb_bvh_params_default(ptb_bvh_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof *p);
    p->max_leaf = 4;
    p->pad_rel = 1e-4f;
    p->n_bins = 16;
    p->smem_nodes = 1024;
    p->traverse_cost = 1.2f;
}
