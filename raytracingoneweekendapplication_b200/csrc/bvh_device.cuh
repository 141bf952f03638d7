// bvh_device.cuh — the scene-upload path that runs on the GPU (SURVEY 8f rank 1).
//
// Replaces, for big scenes, what the reference does in bvh_node's constructor (bvh.h:13-45:
// recursive sort + median split on the host) and what the host path of rt_upload_scene does
// (bake transforms, binned-SAH build, derive the device records on the CPU): the raw ABI
// arrays are copied to the device as they are and seven kernels turn them into the arena the
// render kernel reads —
//
//   prim_map_kernel  (scenes with indexed meshes only) primitive -> (world ref, triangle of the mesh):
//                    a cub scan over the per-ref primitive counts, then a binary search per primitive
//   bounds_kernel    per primitive: bake its transform (double), conservative FP32 box, scene bounds
//   morton_kernel    63-bit Morton code of the box centre (21 bits per axis)
//   cub radix sort   (code, primitive) pairs
//   rank kernels     position of every sorted primitive inside the typed array of ITS type
//                    (4 flag + exclusive-scan passes), so that a subtree's primitives of one type
//                    are contiguous — the leaf encoding needs (type, count, first)
//   karras_kernel    the radix tree over the sorted codes (Karras 2012), one thread per
//                    internal node, no synchronisation
//   fit_kernel       bottom-up: boxes, primitive counts, type masks, heights (one atomic
//                    counter per node; the second thread to arrive owns the parent)
//   nodes_kernel     subtrees of <= 4 primitives of one type collapse into ONE leaf; every other
//                    internal node becomes a 64-byte node {L.min,linkL}{L.max,linkR}{R.min}{R.max}
//   prims_kernel     derive the device records (prim_derive.h, bit-identical to the host path) and
//                    write them in leaf order
//
// All of it is streaming, HBM-bound work: every kernel reads and writes each primitive's record
// once, coalesced in sorted order on the write side; algorithmic bytes per primitive are listed
// in DESIGN.md.  The result is an LBVH: built in milliseconds, traced slower than the host's
// SAH tree (measured numbers in DESIGN.md); rt_set_bvh_builder / RT_B200_BVH choose.
// bvh_refit.cuh refits an uploaded tree of either builder from the same inputs (rt_refit_scene).
#pragma once
#include <cub/cub.cuh>

#include <algorithm>
#include <cstring>
#include <thread>

#include <chrono>
#include <cstdlib>
#include <unordered_map>
#include <vector>

#include "bvh_build.h"
#include "prim_derive.h"

namespace rtlbvh {

using rtprep::BakedPrim;
using rtprep::Sources;

#ifndef RT_LBVH_MAX_LEAF
#define RT_LBVH_MAX_LEAF 4
#endif
constexpr int kMaxLeaf = RT_LBVH_MAX_LEAF;

struct Targets {  // arena blocks the device path fills (world part of each typed array)
    float4* nodes;
    float4 *sph, *msph, *quad, *tri, *tri_sh;
    double *sph_d, *msph_d, *quad_d, *tri_d;
    int4 *sph_sh, *msph_sh, *quad_sh;
};

struct Scratch {
    const rt_prim_ref* world;
    Sources src;
    int n;                                 // primitives: world refs with every mesh ref expanded to its triangles
    uint2* prim_map;                       // per primitive: (world ref, triangle of the mesh); null without meshes
    float4 *box_lo, *box_hi;               // per primitive in INPUT order; lo.w = type bits
    unsigned long long *key_in, *key_out;  // Morton codes
    uint32_t *val_in, *val_out;            // primitive index
    uint32_t *flag, *scan, *rank_at;       // per sorted position
    float* cost;                           // per internal node: SAH cost of its best completion
    const int* quad_light;                 // per SOURCE quad: its number in the next-event emitter list (0: none); may be null
    int *left, *right, *parent_int, *parent_leaf, *range_first;
    float4 *nbox_lo, *nbox_hi;             // per internal node; lo.w = count bits, hi.w = type mask | height << 8
    unsigned* visit;
    unsigned* bounds;                      // 6 ordered-uint floats: centroid min xyz, max xyz
    unsigned* counters;                    // [0] nodes emitted, [1] leaves, [2] height of the root, [3] clusters of the cut, [4] rebuilt clusters, [5] their tallest
    void* cub_temp;
    size_t cub_temp_bytes;
};

__device__ __forceinline__ unsigned ordered(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unordered(unsigned u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

__global__ void init_kernel(Scratch W) {
    if (threadIdx.x < 3) W.bounds[threadIdx.x] = 0xffffffffu;
    else if (threadIdx.x < 6) W.bounds[threadIdx.x] = 0u;
    if (threadIdx.x < 8) W.counters[threadIdx.x] = 0u;
}

// primitives of each world ref (a mesh ref stands for its triangles)
__global__ void __launch_bounds__(256) ref_count_kernel(Scratch W, int n_world, uint32_t* count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_world) return;
    const rt_prim_ref r = W.world[i];
    count[i] = r.type == RT_PRIM_MESH ? (uint32_t)W.src.meshes[r.index].n_triangles : 1u;
}
// primitive p lies in the last world ref whose first primitive is <= p (refs of empty meshes share
// their first with the next ref and are skipped by taking the last)
__global__ void __launch_bounds__(256) prim_map_kernel(Scratch W, const uint32_t* ref_first, int n_world) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= W.n) return;
    int lo = 0, hi = n_world - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (ref_first[mid] <= (uint32_t)p) lo = mid;
        else hi = mid - 1;
    }
    W.prim_map[p] = make_uint2((unsigned)lo, (unsigned)p - ref_first[lo]);
}

// the world ref primitive i comes from, and which triangle of it when it is a mesh ref
template <bool MESH>
__device__ __forceinline__ rt_prim_ref world_ref(const Scratch& W, unsigned i, unsigned* local) {
    if (!MESH) {
        *local = 0;
        return W.world[i];
    }
    const uint2 m = W.prim_map[i];
    *local = m.y;
    return W.world[m.x];
}
template <bool MESH>
__device__ __forceinline__ BakedPrim fetch_prim(const Scratch& W, unsigned i) {
    unsigned k;
    const rt_prim_ref r = world_ref<MESH>(W, i, &k);
    if (MESH && r.type == RT_PRIM_MESH) return rtprep::bake_mesh_triangle(W.src, r.index, k, (int)i);
    return rtprep::bake_prim(W.src, r, (int)i);
}

template <bool MESH>
__global__ void __launch_bounds__(256) bounds_kernel(Scratch W) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float c[3] = {0, 0, 0};
    const bool live = i < W.n;
    if (live) {
        const BakedPrim b = fetch_prim<MESH>(W, (unsigned)i);
        float lo[3], hi[3];
        rtprep::prim_bounds(b, lo, hi);
        W.box_lo[i] = make_float4(lo[0], lo[1], lo[2], __uint_as_float(b.dev_type));
        W.box_hi[i] = make_float4(hi[0], hi[1], hi[2], 0.0f);
        for (int k = 0; k < 3; k++) c[k] = 0.5f * (lo[k] + hi[k]);
    }
    // warp-reduce the centroid bounds, one atomic pair per warp and axis
    for (int k = 0; k < 3; k++) {
        unsigned mn = live ? ordered(c[k]) : 0xffffffffu, mx = live ? ordered(c[k]) : 0u;
        mn = __reduce_min_sync(0xffffffffu, mn);
        mx = __reduce_max_sync(0xffffffffu, mx);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&W.bounds[k], mn);
            atomicMax(&W.bounds[3 + k], mx);
        }
    }
}

__device__ __forceinline__ unsigned long long spread21(unsigned v) {  // 21 bits -> every third bit
    unsigned long long x = v & 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void __launch_bounds__(256) morton_kernel(Scratch W) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W.n) return;
    const float4 lo = W.box_lo[i], hi = W.box_hi[i];
    const float c[3] = {0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z)};
    unsigned q[3];
    for (int k = 0; k < 3; k++) {
        const float mn = unordered(W.bounds[k]), mx = unordered(W.bounds[3 + k]);
        const float ext = mx - mn;
        float t = ext > 0.0f ? (c[k] - mn) / ext : 0.0f;
        t = fminf(fmaxf(t, 0.0f), 1.0f);
        q[k] = min(2097151u, (unsigned)(t * 2097152.0f));
    }
    W.key_in[i] = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
    W.val_in[i] = (unsigned)i;
}

// type of the primitive at sorted position k
__device__ __forceinline__ unsigned type_at(const Scratch& W, int k) { return __float_as_uint(W.box_lo[W.val_out[k]].w); }

__global__ void __launch_bounds__(256) flag_kernel(Scratch W, unsigned type) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < W.n) W.flag[k] = type_at(W, k) == type ? 1u : 0u;
}
__global__ void __launch_bounds__(256) pick_rank_kernel(Scratch W, unsigned type) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < W.n && W.flag[k]) W.rank_at[k] = W.scan[k];
}

// length of the common prefix of the codes at sorted positions i and j (ties broken by position)
__device__ __forceinline__ int delta(const unsigned long long* key, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = key[i], b = key[j];
    if (a == b) return 64 + __clz((unsigned)i ^ (unsigned)j);
    return __clzll((long long)(a ^ b));
}

// Karras, "Maximizing Parallelism in the Construction of BVHs, Octrees, and k-d Trees" (2012):
// internal node i covers a range of sorted leaves that starts or ends at i.
__global__ void __launch_bounds__(256) karras_kernel(Scratch W) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = W.n;
    if (i >= n - 1) return;
    const unsigned long long* key = W.key_out;
    const int d = delta(key, n, i, i + 1) - delta(key, n, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = delta(key, n, i, i - d);
    int lmax = 2;
    while (delta(key, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(key, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(key, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(key, n, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int first = min(i, j), last = max(i, j);
    const int lc = first == gamma ? ~gamma : gamma;
    const int rc = last == gamma + 1 ? ~(gamma + 1) : gamma + 1;
    W.left[i] = lc;
    W.right[i] = rc;
    W.range_first[i] = first;
    if (lc < 0) W.parent_leaf[gamma] = i; else W.parent_int[gamma] = i;
    if (rc < 0) W.parent_leaf[gamma + 1] = i; else W.parent_int[gamma + 1] = i;
    if (i == 0) W.parent_int[0] = -1;
    W.visit[i] = 0u;
}

struct NodeInfo {
    float lo[3], hi[3];
    unsigned count, mask, height;
    float cost;    // SAH cost of the best way to finish this subtree (leaf or split), times the root-independent 1/area factor left out
    bool as_leaf;  // ... and whether that best way is ONE leaf
};
__device__ __forceinline__ float box_area(const float lo[3], const float hi[3]) {
    const float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    return 2.0f * (dx * dy + dy * dz + dz * dx);
}
// relative intersection cost of the primitive types, as the host builder's rtbvh::Prim::cost
__device__ __forceinline__ float prim_cost(unsigned type) { return type == rtprep::PREP_SPHERE ? 1.0f : (type == rtprep::PREP_MSPHERE ? 1.2f : 1.3f); }
#ifndef RT_LBVH_TRAV_COST
#define RT_LBVH_TRAV_COST 3.0f
#endif
constexpr float kTravCost = RT_LBVH_TRAV_COST;  // one node visit, in sphere tests (rtbvh::Tuning::trav_cost)
__device__ __forceinline__ NodeInfo child_info(const Scratch& W, int c) {
    NodeInfo r;
    if (c < 0) {
        const unsigned s = W.val_out[~c];
        const float4 lo = W.box_lo[s], hi = W.box_hi[s];
        r.lo[0] = lo.x; r.lo[1] = lo.y; r.lo[2] = lo.z;
        r.hi[0] = hi.x; r.hi[1] = hi.y; r.hi[2] = hi.z;
        r.count = 1u;
        r.mask = 1u << __float_as_uint(lo.w);
        r.height = 0u;
        r.cost = box_area(r.lo, r.hi) * prim_cost(__float_as_uint(lo.w));
        r.as_leaf = true;
    } else {
        // written by another thread of this launch: read through L2
        const float4 lo = __ldcg(W.nbox_lo + c), hi = __ldcg(W.nbox_hi + c);
        r.lo[0] = lo.x; r.lo[1] = lo.y; r.lo[2] = lo.z;
        r.hi[0] = hi.x; r.hi[1] = hi.y; r.hi[2] = hi.z;
        r.count = __float_as_uint(lo.w);
        r.mask = __float_as_uint(hi.w) & 0x0fu;
        r.as_leaf = (__float_as_uint(hi.w) & 0x80u) != 0u;
        r.height = __float_as_uint(hi.w) >> 8;
        r.cost = __ldcg(W.cost + c);
    }
    return r;
}

__global__ void __launch_bounds__(256) fit_kernel(Scratch W) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= W.n) return;
    int p = W.parent_leaf[k];
    while (p >= 0) {
        __threadfence();
        if (atomicAdd(&W.visit[p], 1u) == 0u) return;  // the sibling subtree is not finished: its thread continues
        __threadfence();
        const NodeInfo a = child_info(W, W.left[p]), b = child_info(W, W.right[p]);
        const unsigned height = max(a.height, b.height) + 1u;
        float lo[3], hi[3];
        for (int k = 0; k < 3; k++) { lo[k] = fminf(a.lo[k], b.lo[k]); hi[k] = fmaxf(a.hi[k], b.hi[k]); }
        const unsigned count = a.count + b.count, mask = a.mask | b.mask;
        // surface-area heuristic, bottom-up: one leaf of `count` primitives of one type, or a node
        // visit plus the best of the two subtrees
        const float area = box_area(lo, hi);
        const float split_cost = kTravCost * area + a.cost + b.cost;
        const bool can_leaf = count <= (unsigned)kMaxLeaf && __popc(mask) == 1;
        const float leaf_cost = area * (float)count * prim_cost(31u - __clz(mask));
        const bool as_leaf = can_leaf && leaf_cost <= split_cost;
        __stcg(W.cost + p, as_leaf ? leaf_cost : split_cost);
        __stcg(W.nbox_lo + p, make_float4(lo[0], lo[1], lo[2], __uint_as_float(count)));
        __stcg(W.nbox_hi + p, make_float4(hi[0], hi[1], hi[2], __uint_as_float(mask | (as_leaf ? 0x80u : 0u) | (height << 8))));
        if (p == 0) W.counters[2] = height;
        p = W.parent_int[p];
    }
}

// A subtree becomes ONE leaf where the SAH says so (and the leaf encoding allows it: <= kMaxLeaf
// primitives of one type).  Nodes below such a subtree root are never referenced.
__device__ __forceinline__ bool collapsible(const NodeInfo& v) { return v.as_leaf; }

constexpr float kClusterTravCost = 1.0f;  // the host builder's rtbvh::Tuning::trav_cost (its cost is normalised by the parent's area)
#include "bvh_cluster_sah.cuh"

__global__ void __launch_bounds__(256) nodes_kernel(Scratch W, Targets T) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= W.n - 1) return;
    const NodeInfo me = child_info(W, i);
    if (collapsible(me)) return;  // lives on as a leaf link in an ancestor
    float4 out[4];
    int links[2];
    unsigned leaves = 0;
    for (int side = 0; side < 2; side++) {
        const int c = side == 0 ? W.left[i] : W.right[i];
        const NodeInfo v = child_info(W, c);
        if (c < 0) {
            links[side] = rtprep::leaf_link(31u - __clz(v.mask), 1u, W.rank_at[~c]);
            leaves++;
        } else if (collapsible(v)) {
            links[side] = rtprep::leaf_link(31u - __clz(v.mask), v.count, W.rank_at[W.range_first[c]]);
            leaves++;
        } else {
            links[side] = c;
        }
        float lo[3], hi[3];
        rtprep::pad_box(v.lo, v.hi, lo, hi);
        out[2 * side] = make_float4(lo[0], lo[1], lo[2], 0.0f);
        out[2 * side + 1] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    }
    out[0].w = __int_as_float(links[0]);
    out[1].w = __int_as_float(links[1]);
    float4* dst = T.nodes + 4 * (size_t)i;
    dst[0] = out[0]; dst[1] = out[1]; dst[2] = out[2]; dst[3] = out[3];
    atomicAdd(&W.counters[0], 1u);
    if (leaves) atomicAdd(&W.counters[1], leaves);
}

// ---- hybrid top levels (HLBVH): the radix tree is cut where subtrees drop to <= max_count
// primitives; the cut ("clusters": a few thousand boxes) goes to the host, which builds the TOP of
// the tree over them with the same binned-SAH builder the host path uses, and comes back as a few
// thousand 64-byte nodes whose leaves link into the radix tree.  The Morton order decides only
// the small-scale structure; the large-scale structure, where LBVH trees lose most, is SAH.
struct Cluster {
    float lo[3];
    int link;  // what a top-tree leaf points at: a radix-tree node (>= 0) or a leaf link (< 0)
    float hi[3];
    unsigned count;
};

__global__ void __launch_bounds__(256) clusters_kernel(Scratch W, unsigned max_count, Cluster* out, unsigned cap) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = W.n;
    if (idx >= 2 * n - 1) return;
    int parent, me;
    if (idx < n - 1) { me = idx; parent = W.parent_int[idx]; }
    else { me = ~(idx - (n - 1)); parent = W.parent_leaf[idx - (n - 1)]; }
    const NodeInfo v = child_info(W, me);
    if (v.count > max_count) return;
    if (parent >= 0 && __float_as_uint(W.nbox_lo[parent].w) <= max_count) return;  // an ancestor is the cluster
    const unsigned slot = atomicAdd(&W.counters[3], 1u);
    atomicMax(&W.counters[2], v.height);  // re-used below as "tallest cluster" (the caller reads the root height first)
    if (slot >= cap) return;
    Cluster c;
    for (int k = 0; k < 3; k++) { c.lo[k] = v.lo[k]; c.hi[k] = v.hi[k]; }
    c.count = v.count;
    if (me < 0) c.link = rtprep::leaf_link(31u - __clz(v.mask), 1u, W.rank_at[~me]);
    else if (collapsible(v)) c.link = rtprep::leaf_link(31u - __clz(v.mask), v.count, W.rank_at[W.range_first[me]]);
    else c.link = me;
    out[slot] = c;
}

__device__ __forceinline__ float4 f4(rtprep::F4 v) { return make_float4(v.x, v.y, v.z, v.w); }
__device__ __forceinline__ int4 i4(rtprep::I4 v) { return make_int4(v.x, v.y, v.z, v.w); }

template <bool MESH>
__global__ void __launch_bounds__(256) prims_kernel(Scratch W, Targets T) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= W.n) return;
    const unsigned s = W.val_out[k];
    const BakedPrim b = fetch_prim<MESH>(W, s);
    const size_t r = W.rank_at[k];
    if (b.dev_type == rtprep::PREP_TRI) {
        const rtprep::TriRec v = rtprep::make_triangle(b);
        for (int q = 0; q < 3; q++) T.tri[3 * r + q] = f4(v.t[q]);
        for (int q = 0; q < 9; q++) T.tri_d[9 * r + q] = v.d[q];
        for (int q = 0; q < 3; q++) T.tri_sh[3 * r + q] = f4(v.sh[q]);
    } else if (b.dev_type == rtprep::PREP_QUAD) {
        const rtprep::QuadRec v = rtprep::make_quad(b);
        for (int q = 0; q < 3; q++) T.quad[3 * r + q] = f4(v.q[q]);
        for (int q = 0; q < 12; q++) T.quad_d[12 * r + q] = v.d[q];
        int4 sh = i4(v.sh);
        if (W.quad_light) {
            unsigned local;
            sh.w = W.quad_light[world_ref<MESH>(W, s, &local).index];
        }
        T.quad_sh[r] = sh;
    } else if (b.dev_type == rtprep::PREP_SPHERE) {
        const rtprep::SphereRec v = rtprep::make_sphere(b);
        T.sph[r] = f4(v.g);
        for (int q = 0; q < 4; q++) T.sph_d[4 * r + q] = v.d[q];
        T.sph_sh[r] = i4(v.sh);
    } else {
        const rtprep::MSphereRec v = rtprep::make_msphere(b);
        T.msph[2 * r] = f4(v.g0);
        T.msph[2 * r + 1] = f4(v.g1);
        for (int q = 0; q < 8; q++) T.msph_d[8 * r + q] = v.d[q];
        T.msph_sh[r] = i4(v.sh);
    }
}

// ---- host side ---------------------------------------------------------------------------------
constexpr unsigned kMaxClusters = 16384;  // capacity of the cut handed to the host (and of the top tree)

struct ScratchPlan {
    size_t size = 0;
    size_t add(size_t bytes) {
        size_t off = (size + 255) & ~(size_t)255;
        size = off + (bytes ? bytes : 16);
        return off;
    }
};

// One array behind the meshes (positions, indices, uvs or uv_indices), copied once however many meshes share it.
struct MeshArray {
    const void* host;
    size_t bytes, off;
};

struct Layout {
    size_t world, spheres, quads, triangles, xforms;
    size_t box_lo, box_hi, key_in, key_out, val_in, val_out, flag, scan, rank_at, left, right, parent_int, parent_leaf, range_first,
        nbox_lo, nbox_hi, visit, bounds, counters, cub_temp, clusters, cost, quad_light;
    size_t meshes, ref_count, ref_first, prim_map;
    std::vector<MeshArray> mesh_arrays;
    std::vector<int> mesh_slots;  // per mesh: positions, indices, uvs, uv_indices -> mesh_arrays (-1: none)
    size_t largest_input;         // biggest single host array copied in (decides whether the pinned ring is worth it)
    size_t cub_temp_bytes, total;
};

// The raw ABI arrays of `sc` and, with meshes, the primitive map: the inputs of both the build and the refit
// (bvh_refit.cuh).  `n` primitives: the world refs with every mesh ref expanded (validate_scene counted them).
inline void plan_inputs(ScratchPlan& p, Layout& L, const rt_scene_desc* sc, int n_prims) {
    const size_t n = (size_t)n_prims, n_world = (size_t)sc->n_world;
    L.world = p.add(n_world * sizeof(rt_prim_ref));
    L.spheres = p.add((size_t)sc->n_spheres * sizeof(rt_sphere));
    L.quads = p.add((size_t)sc->n_quads * sizeof(rt_quad));
    L.triangles = p.add((size_t)sc->n_triangles * sizeof(rt_triangle));
    L.xforms = p.add((size_t)sc->n_xforms * sizeof(rt_xform));
    L.largest_input = std::max({(size_t)sc->n_spheres * sizeof(rt_sphere), (size_t)sc->n_quads * sizeof(rt_quad),
                                (size_t)sc->n_triangles * sizeof(rt_triangle)});
    const bool meshes = sc->n_meshes > 0;
    L.meshes = p.add((size_t)sc->n_meshes * sizeof(rt_mesh));
    if (meshes) {
        std::unordered_map<const void*, int> seen;
        auto slot = [&](const void* host, size_t bytes) {
            if (!host || !bytes) return -1;
            auto it = seen.find(host);
            if (it != seen.end()) {
                MeshArray& a = L.mesh_arrays[(size_t)it->second];
                a.bytes = std::max(a.bytes, bytes);
                return it->second;
            }
            seen.emplace(host, (int)L.mesh_arrays.size());
            L.mesh_arrays.push_back(MeshArray{host, bytes, 0});
            return (int)L.mesh_arrays.size() - 1;
        };
        for (int i = 0; i < sc->n_meshes; i++) {
            const rt_mesh& m = sc->meshes[i];
            const size_t t3 = (size_t)m.n_triangles * 3 * sizeof(uint32_t);
            L.mesh_slots.push_back(slot(m.positions, (size_t)m.n_vertices * 3 * sizeof(float)));
            L.mesh_slots.push_back(slot(m.indices, t3));
            L.mesh_slots.push_back(slot(m.uvs, (size_t)m.n_uvs * 2 * sizeof(float)));
            L.mesh_slots.push_back(slot(m.uv_indices, t3));
        }
        for (MeshArray& a : L.mesh_arrays) {
            a.off = p.add(a.bytes);
            L.largest_input = std::max(L.largest_input, a.bytes);
        }
    }
    L.ref_count = p.add(meshes ? n_world * 4 : 0);
    L.ref_first = p.add(meshes ? n_world * 4 : 0);
    L.prim_map = p.add(meshes ? n * 8 : 0);
}

inline Layout plan_scratch(const rt_scene_desc* sc, int n_prims) {
    Layout L{};
    ScratchPlan p;
    const size_t n = (size_t)n_prims, n_world = (size_t)sc->n_world;
    plan_inputs(p, L, sc, n_prims);
    L.box_lo = p.add(n * 16); L.box_hi = p.add(n * 16);
    L.key_in = p.add(n * 8); L.key_out = p.add(n * 8);
    L.val_in = p.add(n * 4); L.val_out = p.add(n * 4);
    L.flag = p.add(n * 4); L.scan = p.add(n * 4); L.rank_at = p.add(n * 4); L.cost = p.add(n * 4);
    L.left = p.add(n * 4); L.right = p.add(n * 4); L.parent_int = p.add(n * 4); L.parent_leaf = p.add(n * 4); L.range_first = p.add(n * 4);
    L.nbox_lo = p.add(n * 16); L.nbox_hi = p.add(n * 16);
    L.visit = p.add(n * 4);
    L.bounds = p.add(64); L.counters = p.add(64);
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, 63);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)std::max(n, n_world));
    L.cub_temp_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
    L.cub_temp = p.add(L.cub_temp_bytes);
    L.clusters = p.add((size_t)kMaxClusters * sizeof(Cluster));
    L.quad_light = p.add((size_t)sc->n_quads * sizeof(int));
    L.total = p.size;
    return L;
}

// Host -> device copy of a big PAGEABLE array.  cudaMemcpyAsync from pageable memory is staged by
// the driver on one thread (~10 GB/s measured on this box); here `kCopyWorkers` host threads copy
// 4 MB chunks into pinned buffers (two per worker) and enqueue the DMA of each chunk themselves, so
// that staging and PCIe transfer overlap and the staging itself runs on several cores.
constexpr size_t kCopyChunk = 4u << 20;
constexpr int kCopyWorkers = 4;
constexpr size_t kCopyRingBytes = kCopyChunk * 2 * kCopyWorkers;

struct CopyRing {
    unsigned char* pinned = nullptr;  // kCopyRingBytes
    cudaEvent_t done[2 * kCopyWorkers] = {};
    bool ready = false;
    cudaError_t init() {
        if (ready) return cudaSuccess;
        cudaError_t e = cudaHostAlloc((void**)&pinned, kCopyRingBytes, cudaHostAllocDefault);
        if (e != cudaSuccess) return e;
        for (auto& ev : done)
            if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
        ready = true;
        return cudaSuccess;
    }
    void release() {
        if (pinned) cudaFreeHost(pinned);
        pinned = nullptr;
        if (ready) for (auto& ev : done) cudaEventDestroy(ev);
        ready = false;
    }
};

inline cudaError_t copy_in(void* dst, const void* src, size_t bytes, cudaStream_t stream, CopyRing& ring, int device) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < 4 * kCopyChunk || !ring.ready) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
    const size_t n_chunks = (bytes + kCopyChunk - 1) / kCopyChunk;
    cudaError_t err[kCopyWorkers];
    auto work = [&](int w) {
        err[w] = cudaSetDevice(device);
        bool used[2] = {false, false};
        for (size_t c = (size_t)w, k = 0; c < n_chunks && err[w] == cudaSuccess; c += kCopyWorkers, k++) {
            const int slot = 2 * w + (int)(k & 1);
            unsigned char* buf = ring.pinned + (size_t)slot * kCopyChunk;
            if (used[k & 1]) err[w] = cudaEventSynchronize(ring.done[slot]);  // the DMA that last read this buffer
            if (err[w] != cudaSuccess) break;
            const size_t off = c * kCopyChunk, len = std::min(kCopyChunk, bytes - off);
            std::memcpy(buf, (const unsigned char*)src + off, len);
            err[w] = cudaMemcpyAsync((unsigned char*)dst + off, buf, len, cudaMemcpyHostToDevice, stream);
            if (err[w] == cudaSuccess) err[w] = cudaEventRecord(ring.done[slot], stream);
            used[k & 1] = true;
        }
        // the buffers must not be reused by the next copy_in before their DMA finished
        for (int b = 0; b < 2 && err[w] == cudaSuccess; b++)
            if (used[b]) err[w] = cudaEventSynchronize(ring.done[2 * w + b]);
    };
    std::thread pool[kCopyWorkers - 1];
    for (int w = 1; w < kCopyWorkers; w++) pool[w - 1] = std::thread(work, w);
    work(0);
    for (auto& t : pool) t.join();
    for (int w = 0; w < kCopyWorkers; w++)
        if (err[w] != cudaSuccess) return err[w];
    return cudaSuccess;
}

struct BuildResult {
    unsigned nodes = 0, leaves = 0, depth = 0;
    size_t bytes_in = 0;     // host -> device bytes: the raw arrays, the mesh table, the SAH top levels
    int root = 0;            // index of the root node in the node array
    unsigned top_nodes = 0;  // nodes of the SAH top tree appended after the n - 1 radix-tree slots (0: pure LBVH)
    unsigned rebuilt_clusters = 0;
    float ms_copy_in = 0, ms_build = 0, ms_emit = 0, ms_top = 0;
};

// Copies the raw arrays of `sc` (the plan_inputs part of `L`) into `scratch` on `stream`, adding the bytes to `bytes_in`.
inline cudaError_t copy_inputs(const rt_scene_desc* sc, unsigned char* scratch, const Layout& L, cudaStream_t stream, CopyRing& ring,
                               int device, size_t& bytes_in) {
    auto at = [&](size_t off) { return scratch + off; };
    cudaError_t e;
#define RT_COPY_IN(field, ptr, count, type)                                                                                   \
    if ((count) > 0) {                                                                                                        \
        if ((e = copy_in(at(L.field), ptr, (size_t)(count) * sizeof(type), stream, ring, device)) != cudaSuccess) return e;  \
        bytes_in += (size_t)(count) * sizeof(type);                                                                           \
    }
    RT_COPY_IN(world, sc->world, sc->n_world, rt_prim_ref)
    RT_COPY_IN(spheres, sc->spheres, sc->n_spheres, rt_sphere)
    RT_COPY_IN(quads, sc->quads, sc->n_quads, rt_quad)
    RT_COPY_IN(triangles, sc->triangles, sc->n_triangles, rt_triangle)
    RT_COPY_IN(xforms, sc->xforms, sc->n_xforms, rt_xform)
    if (sc->n_meshes > 0) {
        // each distinct mesh array once, then the mesh table with its pointers moved to those copies
        for (const MeshArray& a : L.mesh_arrays) {
            if ((e = copy_in(at(a.off), a.host, a.bytes, stream, ring, device)) != cudaSuccess) return e;
            bytes_in += a.bytes;
        }
        std::vector<rt_mesh> table(sc->meshes, sc->meshes + sc->n_meshes);
        auto dev = [&](int slot) -> const void* { return slot < 0 ? nullptr : at(L.mesh_arrays[(size_t)slot].off); };
        for (size_t i = 0; i < table.size(); i++) {
            table[i].positions = (const float*)dev(L.mesh_slots[4 * i]);
            table[i].indices = (const uint32_t*)dev(L.mesh_slots[4 * i + 1]);
            table[i].uvs = (const float*)dev(L.mesh_slots[4 * i + 2]);
            table[i].uv_indices = (const uint32_t*)dev(L.mesh_slots[4 * i + 3]);
        }
        // pageable source: cudaMemcpyAsync has staged it by the time it returns, so `table` may go
        RT_COPY_IN(meshes, table.data(), sc->n_meshes, rt_mesh)
    }
#undef RT_COPY_IN
    return cudaSuccess;
}

// The copied inputs as the kernels read them: world list, typed sources, primitive count and map
inline Scratch input_view(const rt_scene_desc* sc, int n, unsigned char* scratch, const Layout& L) {
    Scratch W{};
    auto at = [&](size_t off) { return scratch + off; };
    W.world = (const rt_prim_ref*)at(L.world);
    W.src = Sources{(const rt_sphere*)at(L.spheres), (const rt_quad*)at(L.quads), (const rt_triangle*)at(L.triangles),
                    (const rt_xform*)at(L.xforms), (const rt_mesh*)at(L.meshes)};
    W.n = n;
    W.prim_map = sc->n_meshes > 0 ? (uint2*)at(L.prim_map) : nullptr;
    return W;
}

// Scenes with meshes: primitive -> (world ref, triangle of the mesh), from a scan over the per-ref primitive counts
inline cudaError_t map_prims(const Scratch& W, int n_world, unsigned char* scratch, const Layout& L, void* cub_temp, size_t cub_temp_bytes,
                             cudaStream_t stream) {
    const int tpb = 256;
    uint32_t* count = (uint32_t*)(scratch + L.ref_count);
    uint32_t* first = (uint32_t*)(scratch + L.ref_first);
    ref_count_kernel<<<(n_world + tpb - 1) / tpb, tpb, 0, stream>>>(W, n_world, count);
    cudaError_t e = cub::DeviceScan::ExclusiveSum(cub_temp, cub_temp_bytes, count, first, n_world, stream);
    if (e != cudaSuccess) return e;
    prim_map_kernel<<<(W.n + tpb - 1) / tpb, tpb, 0, stream>>>(W, first, n_world);
    return cudaSuccess;
}

// Copies the raw arrays of `sc` into `scratch` and runs the build of its `n` primitives (world refs
// with the mesh refs expanded) on `stream`.  `T` points into the scene arena.  Returns a
// cudaError_t-compatible code (0 = success).  The mesh indices must have been checked.
inline cudaError_t build_on_device(const rt_scene_desc* sc, int n, unsigned char* scratch, const Layout& L, const Targets& T,
                                   cudaStream_t stream, CopyRing& ring, int device, bool hybrid_top, const int* quad_light,
                                   BuildResult& out) {
    const int n_world = sc->n_world;
    const bool meshes = sc->n_meshes > 0;
    auto at = [&](size_t off) { return scratch + off; };
    cudaError_t e;
    cudaEvent_t ev[4];
    for (auto& v : ev) if ((e = cudaEventCreate(&v)) != cudaSuccess) return e;
    cudaEventRecord(ev[0], stream);
    if ((e = copy_inputs(sc, scratch, L, stream, ring, device, out.bytes_in)) != cudaSuccess) return e;
    if (quad_light) {
        if ((e = copy_in(at(L.quad_light), quad_light, (size_t)sc->n_quads * sizeof(int), stream, ring, device)) != cudaSuccess) return e;
        out.bytes_in += (size_t)sc->n_quads * sizeof(int);
    }
    cudaEventRecord(ev[1], stream);
    Scratch W = input_view(sc, n, scratch, L);
    W.box_lo = (float4*)at(L.box_lo); W.box_hi = (float4*)at(L.box_hi);
    W.key_in = (unsigned long long*)at(L.key_in); W.key_out = (unsigned long long*)at(L.key_out);
    W.val_in = (uint32_t*)at(L.val_in); W.val_out = (uint32_t*)at(L.val_out);
    W.flag = (uint32_t*)at(L.flag); W.scan = (uint32_t*)at(L.scan); W.rank_at = (uint32_t*)at(L.rank_at);
    W.cost = (float*)at(L.cost);
    W.quad_light = quad_light ? (const int*)at(L.quad_light) : nullptr;
    W.left = (int*)at(L.left); W.right = (int*)at(L.right); W.parent_int = (int*)at(L.parent_int);
    W.parent_leaf = (int*)at(L.parent_leaf); W.range_first = (int*)at(L.range_first);
    W.nbox_lo = (float4*)at(L.nbox_lo); W.nbox_hi = (float4*)at(L.nbox_hi);
    W.visit = (unsigned*)at(L.visit);
    W.bounds = (unsigned*)at(L.bounds); W.counters = (unsigned*)at(L.counters);
    W.cub_temp = at(L.cub_temp); W.cub_temp_bytes = L.cub_temp_bytes;

    const int tpb = 256, gn = (n + tpb - 1) / tpb, gi = (n - 1 + tpb - 1) / tpb;
    init_kernel<<<1, 32, 0, stream>>>(W);
    size_t tb = W.cub_temp_bytes;
    if (meshes) {
        if ((e = map_prims(W, n_world, scratch, L, W.cub_temp, tb, stream)) != cudaSuccess) return e;
        bounds_kernel<true><<<gn, tpb, 0, stream>>>(W);
    } else {
        bounds_kernel<false><<<gn, tpb, 0, stream>>>(W);
    }
    morton_kernel<<<gn, tpb, 0, stream>>>(W);
    tb = W.cub_temp_bytes;
    if ((e = cub::DeviceRadixSort::SortPairs(W.cub_temp, tb, W.key_in, W.key_out, W.val_in, W.val_out, n, 0, 63, stream)) != cudaSuccess) return e;
    karras_kernel<<<gi, tpb, 0, stream>>>(W);
    fit_kernel<<<gn, tpb, 0, stream>>>(W);
    if (hybrid_top) {
        // SAH rebuild of every subtree of 3..kClusterMax primitives (one warp each); permutes the
        // sorted order inside the clusters, so it runs before the typed ranks are taken
        int* roots = (int*)W.scan;  // free until the rank passes
        cluster_roots_kernel<<<gi, tpb, 0, stream>>>(W, roots, W.counters + 4);
        // a balanced tree has about 2n / kClusterMax clusters; the grid is sized for twice that and surplus
        // warps leave at once.  A degenerate (chain-like) radix tree can have up to n / 3 small clusters: the
        // ones beyond the grid simply keep their radix subtree, which is a valid tree either way
        const int max_clusters = 4 * (n / kClusterMax) + 4;
        cluster_sah_kernel<<<(max_clusters + kClusterWarps - 1) / kClusterWarps, 32 * kClusterWarps, 0, stream>>>(W, roots, W.counters + 4, W.counters + 5);
    }
    for (unsigned t = 0; t < 4; t++) {
        flag_kernel<<<gn, tpb, 0, stream>>>(W, t);
        tb = W.cub_temp_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(W.cub_temp, tb, W.flag, W.scan, n, stream)) != cudaSuccess) return e;
        pick_rank_kernel<<<gn, tpb, 0, stream>>>(W, t);
    }
    cudaEventRecord(ev[2], stream);
    nodes_kernel<<<gi, tpb, 0, stream>>>(W, T);
    if (meshes) prims_kernel<true><<<gn, tpb, 0, stream>>>(W, T);
    else prims_kernel<false><<<gn, tpb, 0, stream>>>(W, T);
    cudaEventRecord(ev[3], stream);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    unsigned c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if ((e = cudaMemcpyAsync(c, W.counters, sizeof c, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    out.nodes = c[0];
    out.leaves = c[1];
    const unsigned rebuilt_tallest = c[5];
    out.depth = c[2] + rebuilt_tallest;  // an upper bound: radix-tree height + the tallest rebuilt cluster
    out.rebuilt_clusters = c[4];
    out.root = 0;
    out.top_nodes = 0;
    // ---- SAH top levels over the cut of the radix tree ------------------------------------------
    const unsigned max_count = std::max<unsigned>((unsigned)kClusterMax, (unsigned)(2ull * (unsigned long long)n / (kMaxClusters / 2)));
    if (hybrid_top && (unsigned)n > 4 * max_count) {
        auto t0 = std::chrono::steady_clock::now();
        Cluster* d_clusters = (Cluster*)at(L.clusters);
        const unsigned zero[2] = {0u, 0u};
        if ((e = cudaMemcpyAsync(W.counters + 2, zero, sizeof zero, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
        clusters_kernel<<<(2 * n - 1 + tpb - 1) / tpb, tpb, 0, stream>>>(W, max_count, d_clusters, kMaxClusters);
        if ((e = cudaMemcpyAsync(c, W.counters, sizeof c, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
        const unsigned n_clusters = c[3], tallest = c[2];
        if (n_clusters >= 2 && n_clusters <= kMaxClusters) {
            std::vector<Cluster> cl(n_clusters);
            if ((e = cudaMemcpy(cl.data(), d_clusters, n_clusters * sizeof(Cluster), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
            std::vector<rtbvh::Prim> items(n_clusters);
            for (unsigned i = 0; i < n_clusters; i++) {
                rtbvh::Prim& p = items[i];
                for (int k = 0; k < 3; k++) { p.box.lo[k] = cl[i].lo[k]; p.box.hi[k] = cl[i].hi[k]; p.centroid[k] = 0.5f * (cl[i].lo[k] + cl[i].hi[k]); }
                p.type = 0;
                p.index = i;
                p.cost = (float)cl[i].count;
            }
            rtbvh::Tuning tune;
            tune.max_leaf = 1;
            rtbvh::Result top;
            rtbvh::build_bvh(items, top, tune, 1);
            // leaves of the top tree are (type 0, count 1, first = position in top.order): point them at the clusters
            const int base = n - 1;
            auto relink = [&](int32_t link) -> int32_t {
                if (link >= 0) return link + base;
                const uint32_t first = (~(uint32_t)link) & 0x01ffffffu;
                return cl[top.order[first]].link;
            };
            for (rtbvh::Node& nd : top.nodes) { nd.llink = relink(nd.llink); nd.rlink = relink(nd.rlink); }
            if (top.root >= 0 && !top.nodes.empty()) {
                // on `stream` and waited for: a plain cudaMemcpy from pageable memory returns once the data is staged, and
                // the render kernels run on a non-blocking stream that the legacy stream does not order against
                if ((e = cudaMemcpyAsync(T.nodes + 4 * (size_t)base, top.nodes.data(), top.nodes.size() * sizeof(rtbvh::Node), cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
                out.bytes_in += top.nodes.size() * sizeof(rtbvh::Node);
                if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
                out.root = top.root + base;
                out.top_nodes = (unsigned)top.nodes.size();
                out.depth = top.depth + tallest + rebuilt_tallest;
                out.nodes += out.top_nodes;
            }
        }
        out.ms_top = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    cudaEventElapsedTime(&out.ms_copy_in, ev[0], ev[1]);
    cudaEventElapsedTime(&out.ms_build, ev[1], ev[2]);
    cudaEventElapsedTime(&out.ms_emit, ev[2], ev[3]);
    for (auto& v : ev) cudaEventDestroy(v);
    return cudaSuccess;
}

}  // namespace rtlbvh
