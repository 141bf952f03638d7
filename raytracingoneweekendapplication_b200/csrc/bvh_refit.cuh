// bvh_refit.cuh — rt_refit_scene on the GPU: the uploaded tree keeps its topology and leaf order, the records are
// re-baked from a changed description of the same structure and the node boxes are recomputed (DESIGN.md section 10c).
// One path for host-built and device-built trees:
//
//   inputs              the raw arrays are copied in as the device build copies them (copy_inputs, map_prims)
//   refit_check_kernel  read only: every world record slot names its canonical primitive in its shading word; the
//                       primitive of the NEW description must have the slot's device type, else the refit is refused
//                       before anything in the arena is written
//   refit_bake_kernel   the record of that primitive, written in place (prim_derive.h: bit-identical to an upload),
//                       and its conservative FP32 box
//   refit_walk_kernel   once per uploaded tree: breadth-first order of the nodes REACHABLE from the root, one launch
//                       per level.  A device-built tree has node slots nothing links to (radix nodes below a collapsed
//                       subtree, radix nodes above the SAH top levels) that hold stale bytes, so the tree is walked
//                       from the root, never scanned slot by slot
//   refit_nodes_kernel  bottom-up, one launch per level: each node's two child boxes (a leaf's record boxes or a
//                       child node's union), padded and written in the paired layout
//
// Included by rt_b200.cu after pair_node.
#pragma once
#include "buffer.h"
#include "bvh_device.cuh"

namespace rtlbvh {

// World record slots of the arena.  Slot k of the n world primitives has type t for base[t] <= k < base[t + 1] and is
// record k - base[t] of that type's array (the boundary records follow the world records in each array).
struct RefitSlots {
    Targets T;
    unsigned base[5];
    // device-built trees: per SOURCE quad its number in the next-event emitter list (0: none), as prims_kernel reads
    // it; null for host-built trees, whose emitter numbers belong to the canonical slot and stay with it
    const int* quad_light;
};

// the type of world slot k and its record number r in that type's array
__device__ __forceinline__ unsigned slot_type(const RefitSlots& R, unsigned k, unsigned* r) {
    const unsigned b1 = R.base[1], b2 = R.base[2], b3 = R.base[3];
    const unsigned t = (k >= b1 ? 1u : 0u) + (k >= b2 ? 1u : 0u) + (k >= b3 ? 1u : 0u);
    *r = k - (t == 0 ? 0u : (t == 1 ? b1 : (t == 2 ? b2 : b3)));
    return t;
}
// canonical id of the primitive record r of type t was derived from (its shading word)
__device__ __forceinline__ unsigned slot_prim(const RefitSlots& R, unsigned t, unsigned r) {
    if (t == rtprep::PREP_SPHERE) return (unsigned)R.T.sph_sh[r].z;
    if (t == rtprep::PREP_MSPHERE) return (unsigned)R.T.msph_sh[r].z;
    if (t == rtprep::PREP_QUAD) return (unsigned)R.T.quad_sh[r].z;
    return __float_as_uint(R.T.tri_sh[3 * (size_t)r + 2].z);
}

// bad: the smallest (canonical id << 4 | slot type << 2 | new type) of a slot whose primitive changed type (~0u: none)
template <bool MESH>
__global__ void __launch_bounds__(256) refit_check_kernel(Scratch W, RefitSlots R, unsigned* bad) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= W.n) return;
    unsigned r;
    const unsigned t = slot_type(R, (unsigned)k, &r);
    const unsigned id = slot_prim(R, t, r);
    const BakedPrim b = fetch_prim<MESH>(W, id);
    if (b.dev_type != t) atomicMin(bad, id << 4 | t << 2 | b.dev_type);
}

template <bool MESH>
__global__ void __launch_bounds__(256) refit_bake_kernel(Scratch W, RefitSlots R) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= W.n) return;
    unsigned r;
    const unsigned t = slot_type(R, (unsigned)k, &r);
    const unsigned id = slot_prim(R, t, r);
    const BakedPrim b = fetch_prim<MESH>(W, id);
    float lo[3], hi[3];
    rtprep::prim_bounds(b, lo, hi);
    W.box_lo[k] = make_float4(lo[0], lo[1], lo[2], 0.0f);
    W.box_hi[k] = make_float4(hi[0], hi[1], hi[2], 0.0f);
    // the records as prims_kernel writes them, with the quads' emitter numbers of the list in its uploaded order
    const Targets& T = R.T;
    if (t == rtprep::PREP_TRI) {
        const rtprep::TriRec v = rtprep::make_triangle(b);
        for (int q = 0; q < 3; q++) T.tri[3 * (size_t)r + q] = f4(v.t[q]);
        for (int q = 0; q < 9; q++) T.tri_d[9 * (size_t)r + q] = v.d[q];
        for (int q = 0; q < 3; q++) T.tri_sh[3 * (size_t)r + q] = f4(v.sh[q]);
    } else if (t == rtprep::PREP_QUAD) {
        const rtprep::QuadRec v = rtprep::make_quad(b);
        for (int q = 0; q < 3; q++) T.quad[3 * (size_t)r + q] = f4(v.q[q]);
        for (int q = 0; q < 12; q++) T.quad_d[12 * (size_t)r + q] = v.d[q];
        int4 sh = i4(v.sh);
        if (R.quad_light) {
            unsigned local;
            sh.w = R.quad_light[world_ref<MESH>(W, id, &local).index];
        } else {
            sh.w = T.quad_sh[r].w;
        }
        T.quad_sh[r] = sh;
    } else if (t == rtprep::PREP_SPHERE) {
        const rtprep::SphereRec v = rtprep::make_sphere(b);
        T.sph[r] = f4(v.g);
        for (int q = 0; q < 4; q++) T.sph_d[4 * (size_t)r + q] = v.d[q];
        T.sph_sh[r] = i4(v.sh);
    } else {
        const rtprep::MSphereRec v = rtprep::make_msphere(b);
        T.msph[2 * (size_t)r] = f4(v.g0);
        T.msph[2 * (size_t)r + 1] = f4(v.g1);
        for (int q = 0; q < 8; q++) T.msph_d[8 * (size_t)r + q] = v.d[q];
        T.msph_sh[r] = i4(v.sh);
    }
}

// Level `level` of the breadth-first order: count[l] nodes at level l, stored from sum(count[0 .. l - 1]) on in
// `order`; appends the level's child nodes (at most `cap` positions in all) and records where each child went (-1: a
// leaf).
__global__ void __launch_bounds__(256) refit_walk_kernel(const float4* nodes, int* order, int2* kids, int* count, int level, int cap) {
    int begin = 0;
    for (int l = 0; l < level; l++) begin += count[l];
    const int n = count[level], end = begin + n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int node = order[begin + i];
        const float4 links = nodes[4 * (size_t)node + 3];  // paired layout: {llink, rlink, -, -}
        int kid[2] = {-1, -1};
        for (int side = 0; side < 2; side++) {
            const int link = __float_as_int(side == 0 ? links.x : links.y);
            if (link < 0) continue;
            const int at = end + atomicAdd(&count[level + 1], 1);
            if (at < cap) {
                order[at] = link;
                kid[side] = at;
            }
        }
        kids[begin + i] = make_int2(kid[0], kid[1]);
    }
}

// One level of the bottom-up pass, positions [begin, begin + n) of the breadth-first order.  box: union of each
// node's two children, unpadded, per position (the parent level reads it).
__global__ void __launch_bounds__(256) refit_nodes_kernel(float4* nodes, const int* order, const int2* kids, float4* box_lo, float4* box_hi,
                                                          Scratch W, RefitSlots R, int begin, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int pos = begin + i;
    float4* nd = nodes + 4 * (size_t)order[pos];
    const float4 links = nd[3];
    const int2 kid = kids[pos];
    float4 out[4];
    float all_lo[3], all_hi[3];
    for (int side = 0; side < 2; side++) {
        const int link = __float_as_int(side == 0 ? links.x : links.y);
        float lo[3], hi[3];
        if (link >= 0) {
            const int c = side == 0 ? kid.x : kid.y;
            const float4 a = box_lo[c], b = box_hi[c];
            lo[0] = a.x; lo[1] = a.y; lo[2] = a.z;
            hi[0] = b.x; hi[1] = b.y; hi[2] = b.z;
        } else {
            // leaf link ~(type << 28 | (count - 1) << 25 | first): records first .. first + count - 1 of the type
            const uint32_t v = ~(uint32_t)link;
            const uint32_t type = v >> 28;
            const uint32_t s = (type == 0 ? 0u : (type == 1 ? R.base[1] : (type == 2 ? R.base[2] : R.base[3]))) + (v & 0x1ffffffu);
            const uint32_t cnt = ((v >> 25) & 7u) + 1u;
            for (int k = 0; k < 3; k++) { lo[k] = FLT_MAX; hi[k] = -FLT_MAX; }
            for (uint32_t j = 0; j < cnt; j++) {
                const float4 a = W.box_lo[s + j], b = W.box_hi[s + j];
                lo[0] = fminf(lo[0], a.x); lo[1] = fminf(lo[1], a.y); lo[2] = fminf(lo[2], a.z);
                hi[0] = fmaxf(hi[0], b.x); hi[1] = fmaxf(hi[1], b.y); hi[2] = fmaxf(hi[2], b.z);
            }
        }
        for (int k = 0; k < 3; k++) {
            all_lo[k] = side == 0 ? lo[k] : fminf(all_lo[k], lo[k]);
            all_hi[k] = side == 0 ? hi[k] : fmaxf(all_hi[k], hi[k]);
        }
        float plo[3], phi[3];
        rtprep::pad_box(lo, hi, plo, phi);
        out[2 * side] = make_float4(plo[0], plo[1], plo[2], 0.0f);
        out[2 * side + 1] = make_float4(phi[0], phi[1], phi[2], 0.0f);
    }
    out[0].w = links.x;
    out[1].w = links.y;
    pair_node(out);
    nd[0] = out[0]; nd[1] = out[1]; nd[2] = out[2];
    box_lo[pos] = make_float4(all_lo[0], all_lo[1], all_lo[2], 0.0f);
    box_hi[pos] = make_float4(all_hi[0], all_hi[1], all_hi[2], 0.0f);
}

// ---- host side ---------------------------------------------------------------------------------

// transient work space of one refit: the inputs, a box per world primitive, the check word, the emitter number of each
// source quad, the scan of the mesh refs
inline Layout plan_refit(const rt_scene_desc* sc, int n_prims) {
    Layout L{};
    ScratchPlan p;
    plan_inputs(p, L, sc, n_prims);
    L.box_lo = p.add((size_t)n_prims * 16);
    L.box_hi = p.add((size_t)n_prims * 16);
    L.counters = p.add(64);
    L.quad_light = p.add((size_t)sc->n_quads * sizeof(int));
    L.cub_temp_bytes = 0;
    if (sc->n_meshes > 0)
        cub::DeviceScan::ExclusiveSum(nullptr, L.cub_temp_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, sc->n_world);
    L.cub_temp = p.add(L.cub_temp_bytes);
    L.total = p.size;
    return L;
}

// The uploaded tree as the bottom-up pass visits it, kept from the first refit after an upload to the next upload:
// breadth-first order of the reachable nodes, where each one's child nodes sit in that order, a union box per
// position, and the nodes per level.
struct RefitTree {
    DeviceBuffer<unsigned char> mem;
    int* order = nullptr;
    int2* kids = nullptr;
    float4 *box_lo = nullptr, *box_hi = nullptr;
    int* count = nullptr;        // device: nodes per level
    std::vector<int> levels;     // nodes per level (empty: not derived for the uploaded tree)
};

// Walks the `n_nodes`-slot tree from `root` (a node) on `stream`; at most `max_levels` levels.  Returns false in
// `ok` when the tree does not fit (more reachable nodes than slots, or deeper than max_levels).
inline cudaError_t derive_refit_tree(RefitTree& RT, const float4* nodes, int root, int n_nodes, int max_levels, int sm_count,
                                     cudaStream_t stream, bool& ok) {
    ok = false;
    RT.levels.clear();
    ScratchPlan p;
    const size_t n = (size_t)n_nodes;
    const size_t o_order = p.add(n * 4), o_kids = p.add(n * 8), o_lo = p.add(n * 16), o_hi = p.add(n * 16),
                 o_count = p.add((size_t)(max_levels + 1) * 4);
    cudaError_t e;
    if ((e = RT.mem.reserve(p.size)) != cudaSuccess) return e;
    RT.order = (int*)(RT.mem + o_order);
    RT.kids = (int2*)(RT.mem + o_kids);
    RT.box_lo = (float4*)(RT.mem + o_lo);
    RT.box_hi = (float4*)(RT.mem + o_hi);
    RT.count = (int*)(RT.mem + o_count);
    std::vector<int> count((size_t)max_levels + 1, 0);
    count[0] = 1;
    if ((e = cudaMemcpyAsync(RT.count, count.data(), count.size() * 4, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(RT.order, &root, 4, cudaMemcpyHostToDevice, stream)) != cudaSuccess) return e;
    for (int l = 0; l < max_levels; l++)
        refit_walk_kernel<<<2 * sm_count, 256, 0, stream>>>(nodes, RT.order, RT.kids, RT.count, l, n_nodes);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(count.data(), RT.count, count.size() * 4, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    long long total = 0;
    for (int l = 0; l <= max_levels; l++) total += count[(size_t)l];
    if (count[(size_t)max_levels] != 0 || total > n_nodes) return cudaSuccess;
    for (int l = 0; l < max_levels && count[(size_t)l] > 0; l++) RT.levels.push_back(count[(size_t)l]);
    ok = true;
    return cudaSuccess;
}

// Re-bakes the n world records and refits the tree's boxes, on `stream`.  `W` views the copied inputs of the new
// description (its box and counter fields point into the refit work space).
inline cudaError_t refit_on_device(const Scratch& W, const RefitSlots& R, bool meshes, float4* nodes, const RefitTree& RT, cudaStream_t stream) {
    const int tpb = 256;
    if (W.n > 0) {
        if (meshes) refit_bake_kernel<true><<<(W.n + tpb - 1) / tpb, tpb, 0, stream>>>(W, R);
        else refit_bake_kernel<false><<<(W.n + tpb - 1) / tpb, tpb, 0, stream>>>(W, R);
    }
    int begin = 0;
    for (int c : RT.levels) begin += c;
    for (size_t l = RT.levels.size(); l-- > 0;) {
        const int n = RT.levels[l];
        begin -= n;
        refit_nodes_kernel<<<(n + tpb - 1) / tpb, tpb, 0, stream>>>(nodes, RT.order, RT.kids, RT.box_lo, RT.box_hi, W, R, begin, n);
    }
    return cudaGetLastError();
}

}  // namespace rtlbvh
