// bvh_build.h — host-side binned-SAH BVH2 builder for the flattened scene.
//
// Replaces the reference's build (bvh.h:13-45: sort by bbox.min on the longest axis,
// split at the median, one object per leaf, the single object of an odd span stored as
// both children).  Closest-hit results do not depend on the tree, so the device is free
// to use a better one: 16-bin surface-area heuristic on centroid bounds, leaves of up to
// four primitives OF ONE TYPE (so a leaf's primitives are contiguous in one typed array
// and the type test is per leaf, not per primitive), children stored so that one 64-byte
// node holds both child boxes.
#pragma once
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <thread>
#include <vector>

namespace rtbvh {

struct Box {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX};
    float hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    void grow(const Box& b) {
        for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], b.lo[k]); hi[k] = std::max(hi[k], b.hi[k]); }
    }
    void grow(const float* p) {
        for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], p[k]); hi[k] = std::max(hi[k], p[k]); }
    }
    float area() const {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (dx < 0 || dy < 0 || dz < 0) return 0.0f;
        return 2.0f * (dx * dy + dy * dz + dz * dx);
    }
};

struct Prim {
    Box box;
    float centroid[3];
    uint32_t type;   // device primitive type (PT_*)
    uint32_t index;  // index in the typed source array
    float cost;      // relative intersection cost
};

struct Node {  // 64 B, the device layout
    float lmin[3]; int32_t llink;
    float lmax[3]; int32_t rlink;
    float rmin[3]; float pad0;
    float rmax[3]; float pad1;
};

struct Result {
    std::vector<Node> nodes;
    int32_t root = 0;
    std::vector<uint32_t> order;  // primitive indices (into the input vector) in leaf order
    uint32_t depth = 0, leaves = 0;
};

#ifndef RT_SAH_BINS
#define RT_SAH_BINS 16
#endif
constexpr int kBins = RT_SAH_BINS;
constexpr int kAllAxes = 8192;
struct Tuning {
    int max_leaf = 4;       // primitives per leaf (<= 8, the link encoding has 3 count bits)
    float trav_cost = 1.0f; // cost of one node visit relative to a sphere test
    uint32_t all_axes_max = kAllAxes;  // ranges of at most this many primitives get the full 3-axis search
    size_t shortcut_min = 4096;  // scenes with more primitives than this take the build-time shortcuts (fewer bins for small ranges, pairs become leaves unexamined)
};

// One builder instance fills one Result for the index range it is given; `ids` is shared
// between the instances of a parallel build (they work on disjoint ranges of it).
class Builder {
  public:
    Builder(const std::vector<Prim>& prims, uint32_t* shared_ids, Result& out, Tuning t) : P(prims), ids(shared_ids), R(out), tune(t) {
        type_cursor[0] = type_cursor[1] = type_cursor[2] = type_cursor[3] = 0;
    }
    uint32_t type_cursor[4];

    bool single_type(uint32_t a, uint32_t b) const {
        for (uint32_t i = a + 1; i < b; i++)
            if (P[ids[i]].type != P[ids[a]].type) return false;
        return true;
    }

    int32_t make_leaf(uint32_t a, uint32_t b) {
        uint32_t type = P[ids[a]].type, count = b - a;
        uint32_t first = type_cursor[type];
        type_cursor[type] += count;
        for (uint32_t i = a; i < b; i++) R.order.push_back(ids[i]);
        R.leaves++;
        uint32_t v = (type << 28) | ((count - 1) << 25) | first;
        return (int32_t)~v;
    }

    // Bounds of ids[a,b) and the SAH decision: returns true with `mid` set when the range is to be
    // split (ids partitioned in place), false when it becomes a leaf.
    bool choose_split(uint32_t a, uint32_t b, Box& bounds, uint32_t& mid) {
        Box cb;
        bounds = Box();
        float total_cost = 0;
        for (uint32_t i = a; i < b; i++) {
            bounds.grow(P[ids[i]].box);
            cb.grow(P[ids[i]].centroid);
            total_cost += P[ids[i]].cost;
        }
        const uint32_t n = b - a;
        if (n == 1) return false;
        // two primitives of one type: a leaf costs 2 tests, a split costs a node visit plus (on
        // average) more than one test -- never worth evaluating (and it halves the node count)
        // (only for big scenes, where build time is end-to-end time; small scenes such as the
        // Cornell box measurably prefer the full SAH decision: 1850 vs 1660 Msamples/s)
        if (n == 2 && tune.max_leaf >= 2 && P.size() > tune.shortcut_min && single_type(a, b)) return false;

        int best_axis = -1, best_bin = -1;
        float best_cost = FLT_MAX;
        // small ranges of BIG scenes use fewer bins (most of 16 would be empty and the fixed cost per
        // node dominates the build); small scenes always get the full resolution
        const int nbins = P.size() <= tune.shortcut_min ? kBins : (n < 8 ? 4 : (n < 32 ? 8 : kBins));
        const float parent_area = std::max(bounds.area(), 1e-30f);
        // Large ranges are binned along the longest centroid axis only (the other axes are tried
        // if that one offers no split); ranges of <= kAllAxes primitives get the full 3-axis search.
        // Building is on the scene-upload path (host time is end-to-end time).  The limit was 256 at
        // first ("the top of the tree is where a single axis is almost always the SAH winner"): measured,
        // the full search at the top is worth +3.3 % on C5 (an A/B over Tuning::all_axes_max), and scenes big enough
        // for it to cost build time go to the device builder anyway.
        int order_axes[3] = {0, 1, 2};
        std::sort(order_axes, order_axes + 3, [&](int x, int y) { return cb.hi[x] - cb.lo[x] > cb.hi[y] - cb.lo[y]; });
        for (int ai = 0; ai < 3; ai++) {
            const int axis = order_axes[ai];
            if (ai > 0 && best_axis >= 0 && n > tune.all_axes_max) break;
            float ext = cb.hi[axis] - cb.lo[axis];
            if (!(ext > 0)) continue;
            Box bin_box[kBins];
            float bin_cost[kBins] = {0};
            const float scale = nbins / ext;
            for (uint32_t i = a; i < b; i++) {
                const Prim& p = P[ids[i]];
                int bi = std::min(nbins - 1, std::max(0, (int)((p.centroid[axis] - cb.lo[axis]) * scale)));
                bin_box[bi].grow(p.box);
                bin_cost[bi] += p.cost;
            }
            float right_area[kBins], right_cost[kBins];
            Box acc;
            float c = 0;
            for (int i = nbins - 1; i > 0; i--) {
                acc.grow(bin_box[i]);
                c += bin_cost[i];
                right_area[i] = acc.area();
                right_cost[i] = c;
            }
            acc = Box();
            c = 0;
            for (int i = 0; i < nbins - 1; i++) {
                acc.grow(bin_box[i]);
                c += bin_cost[i];
                if (c == 0 || right_cost[i + 1] == 0) continue;
                float cost = tune.trav_cost + (acc.area() * c + right_area[i + 1] * right_cost[i + 1]) / parent_area;
                if (cost < best_cost) { best_cost = cost; best_axis = axis; best_bin = i; }
            }
        }
        const bool can_leaf = n <= (uint32_t)tune.max_leaf && single_type(a, b);
        if (can_leaf && (best_axis < 0 || total_cost <= best_cost)) return false;

        if (best_axis >= 0) {
            const float ext = cb.hi[best_axis] - cb.lo[best_axis];
            const float scale = nbins / ext;
            const float lo = cb.lo[best_axis];
            const int axis = best_axis, bin = best_bin;
            auto it = std::partition(ids + a, ids + b, [&](uint32_t id) {
                int bi = std::min(nbins - 1, std::max(0, (int)((P[id].centroid[axis] - lo) * scale)));
                return bi <= bin;
            });
            mid = (uint32_t)(it - ids);
        } else {
            mid = a;  // all centroids coincide
        }
        if (mid == a || mid == b) {
            // degenerate (coincident centroids, or mixed types that binning cannot separate):
            // group by type, then halve
            std::stable_sort(ids + a, ids + b, [&](uint32_t x, uint32_t y) { return P[x].type < P[y].type; });
            mid = a + n / 2;
            for (uint32_t i = a + 1; i < b; i++)
                if (P[ids[i]].type != P[ids[i - 1]].type) { mid = i; break; }
        }
        return true;
    }

    static void fill_node(Node& nd, const Box& lb, const Box& rb, int32_t l, int32_t r) {
        const float pad = 1e-6f;
        for (int k = 0; k < 3; k++) {
            // conservative outward rounding so that FP32 slab tests never cull a true hit
            float e = pad * std::max({1.0f, std::fabs(lb.lo[k]), std::fabs(lb.hi[k])});
            nd.lmin[k] = lb.lo[k] - e; nd.lmax[k] = lb.hi[k] + e;
            e = pad * std::max({1.0f, std::fabs(rb.lo[k]), std::fabs(rb.hi[k])});
            nd.rmin[k] = rb.lo[k] - e; nd.rmax[k] = rb.hi[k] + e;
        }
        nd.llink = l;
        nd.rlink = r;
        nd.pad0 = nd.pad1 = 0;
    }

    // sequential build: returns the link of the subtree over ids[a,b) and its bounds
    int32_t build(uint32_t a, uint32_t b, Box& bounds, uint32_t depth) {
        R.depth = std::max(R.depth, depth);
        uint32_t mid = a;
        if (!choose_split(a, b, bounds, mid)) return make_leaf(a, b);
        Box lb, rb;
        int32_t me = (int32_t)R.nodes.size();
        R.nodes.push_back(Node{});
        int32_t l = build(a, mid, lb, depth + 1);
        int32_t r = build(mid, b, rb, depth + 1);
        fill_node(R.nodes[me], lb, rb, l, r);
        return me;
    }

  private:
    const std::vector<Prim>& P;
    uint32_t* ids;
    Result& R;
    Tuning tune;
};

// A finished subtree of the parallel build
struct Subtree {
    Result R;
    uint32_t type_count[4] = {0, 0, 0, 0};
    int32_t link = 0;
    Box bounds;
};

constexpr uint32_t kParallelMin = 2048;  // ranges below this are built by one thread

// shifts a link of a subtree that is being appended after `node_off` nodes and after
// `type_off[t]` primitives of each type
inline int32_t shift_link(int32_t link, int32_t node_off, const uint32_t* type_off) {
    if (link >= 0) return link + node_off;
    uint32_t v = ~(uint32_t)link;
    uint32_t type = v >> 28, rest = v & 0x0e000000u, first = v & 0x01ffffffu;
    return (int32_t)~((type << 28) | rest | (first + type_off[type]));
}

inline void build_parallel(const std::vector<Prim>& P, uint32_t* ids, uint32_t a, uint32_t b, const Tuning& tune, uint32_t depth,
                           int budget, Subtree& out) {
    Builder bd(P, ids, out.R, tune);
    uint32_t mid = a;
    if (budget <= 1 || b - a < kParallelMin) {
        out.link = bd.build(a, b, out.bounds, depth);
        for (int t = 0; t < 4; t++) out.type_count[t] = bd.type_cursor[t];
        return;
    }
    if (!bd.choose_split(a, b, out.bounds, mid)) {
        out.link = bd.make_leaf(a, b);
        for (int t = 0; t < 4; t++) out.type_count[t] = bd.type_cursor[t];
        out.R.depth = depth;
        return;
    }
    Subtree left, right;
    std::thread worker([&]() { build_parallel(P, ids, a, mid, tune, depth + 1, budget / 2, left); });
    build_parallel(P, ids, mid, b, tune, depth + 1, budget - budget / 2, right);
    worker.join();
    // merge: [parent][left nodes][right nodes]; left primitives first in every typed array
    const uint32_t zero[4] = {0, 0, 0, 0};
    const int32_t loff = 1, roff = 1 + (int32_t)left.R.nodes.size();
    out.R.nodes.reserve(1 + left.R.nodes.size() + right.R.nodes.size());
    out.R.nodes.push_back(Node{});
    for (Node n : left.R.nodes) {
        n.llink = shift_link(n.llink, loff, zero);
        n.rlink = shift_link(n.rlink, loff, zero);
        out.R.nodes.push_back(n);
    }
    for (Node n : right.R.nodes) {
        n.llink = shift_link(n.llink, roff, left.type_count);
        n.rlink = shift_link(n.rlink, roff, left.type_count);
        out.R.nodes.push_back(n);
    }
    Builder::fill_node(out.R.nodes[0], left.bounds, right.bounds, shift_link(left.link, loff, zero),
                       shift_link(right.link, roff, left.type_count));
    out.R.order = std::move(left.R.order);
    out.R.order.insert(out.R.order.end(), right.R.order.begin(), right.R.order.end());
    out.R.depth = std::max({depth, left.R.depth, right.R.depth});
    out.R.leaves = left.R.leaves + right.R.leaves;
    for (int t = 0; t < 4; t++) out.type_count[t] = left.type_count[t] + right.type_count[t];
    out.link = 0;
}

// Entry point: SAH BVH over `prims` using up to `threads` host threads (0 = all).
inline void build_bvh(const std::vector<Prim>& prims, Result& out, Tuning tune = Tuning(), int threads = 0) {
    out = Result();
    if (prims.empty()) {
        // one node whose two child boxes are empty; DevScene::n_world == 0 keeps rays away from it
        Node n{};
        for (int k = 0; k < 3; k++) { n.lmin[k] = n.rmin[k] = FLT_MAX; n.lmax[k] = n.rmax[k] = -FLT_MAX; }
        n.llink = n.rlink = 0;
        out.nodes.push_back(n);
        out.root = 0;
        return;
    }
    std::vector<uint32_t> ids(prims.size());
    for (size_t i = 0; i < prims.size(); i++) ids[i] = (uint32_t)i;
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    Subtree top;
    build_parallel(prims, ids.data(), 0, (uint32_t)prims.size(), tune, 1, threads, top);
    out = std::move(top.R);
    out.root = top.link;
}

}  // namespace rtbvh
