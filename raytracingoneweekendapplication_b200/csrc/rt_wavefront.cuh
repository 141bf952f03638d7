// rt_wavefront.cuh — the wavefront formulation of the bounce loop (RT_B200_KERNEL=wf).
//
// BASELINE.json asks for the bounce loop to be "either a wavefront pipeline (raygen ->
// traverse/extend with warp-level ray compaction -> shade/scatter -> accumulate) or a
// persistent megakernel, picked from ncu evidence".  This is the wavefront candidate; the
// megakernel (render_kernel_v2) is the other.  Both trace exactly the same samples (same Philox
// counters, same device functions) and add them to the frame as 64-bit fixed-point sums, so
// their images are interchangeable.
//
// A pool of P path slots lives in HBM as structure-of-arrays (88 B per path).  One bounce of
// the whole pool is three launches:
//   wf_swap     (1 thread)  next active list becomes current, cursors reset
//   wf_extend   persistent warps pull slot ids from the active list; every lane traverses one
//               ray; a warp refills its idle lanes from the list whenever enough of them are idle
//               (the "ray compaction": refilling costs one 32-byte ray load, not a shade phase)
//   wf_shade    one thread per active path: media, hit completion, emission, scatter; a path
//               that continues is appended to the next list, a path that ends is added to the
//               frame and its slot immediately takes the next (pixel, sample) of the stream
// The extend kernel needs few registers (high occupancy hides the node-fetch latency), and no
// lane ever waits for another lane's shading.  The price is ~200 B of path-state traffic per
// ray through L2/HBM.
#pragma once
#include "rt_device.cuh"

namespace rtwf {
using namespace rtdev;

struct Pool {
    float4* ray_o;   // o.xyz, time
    float4* ray_d;   // d.xyz, as_float(origin_prim)
    float4* thr;     // T.xyz, as_float(bounce)
    float4* rad;     // L.xyz, -
    uint2* id;       // pixel, sample
    float4* hit;     // t, as_float(prim), u, v
    uint32_t* list[2];
    // ctr[0] next index of the sample stream, [1] unused, [2] n_active (current),
    // [3] n_active (next), [4] extend cursor, [5] current list (0/1)
    unsigned long long* ctr;
    uint32_t capacity;
};

struct Stream {  // how the global sample stream maps to (pixel, sample); same enumeration idea as v2
    int width, height, max_depth, spp_begin, n_local_samples, sample_stride, sample_offset;
    int tiles_x, tile_size, tile_stride, tile_offset, blocks_per_tile_x, blocks_per_tile_y;
    unsigned long long total;  // pixel_blocks * 32 * n_local_samples
    uint32_t k0, k1;
};

// Decodes stream index g; returns false for the slots of a pixel block that fall outside the frame.
__device__ __forceinline__ bool decode_sample(const Stream& A, unsigned long long g, int& px, int& py, uint32_t& pixel, uint32_t& sample) {
    const unsigned long long per_block = 32ull * (unsigned long long)A.n_local_samples;
    const unsigned long long blk = g / per_block;
    const unsigned r = (unsigned)(g % per_block);
    const unsigned smp = r >> 5, lp = r & 31u;
    const unsigned blocks_per_tile = (unsigned)(A.blocks_per_tile_x * A.blocks_per_tile_y);
    const unsigned local_tile = (unsigned)(blk / blocks_per_tile), in_tile = (unsigned)(blk % blocks_per_tile);
    const unsigned tile = A.tile_offset + local_tile * A.tile_stride;
    px = (int)(tile % A.tiles_x) * A.tile_size + (int)(in_tile % A.blocks_per_tile_x) * 8 + (int)(lp & 7u);
    py = (int)(tile / A.tiles_x) * A.tile_size + (int)(in_tile / A.blocks_per_tile_x) * 4 + (int)(lp >> 3);
    if (px >= A.width || py >= A.height) return false;
    pixel = (uint32_t)(py * A.width + px);
    sample = (uint32_t)(A.spp_begin + A.sample_offset + (int)smp * A.sample_stride);
    return true;
}

// Takes the next valid (pixel, sample) of the stream and writes a fresh camera path into `slot`.
__device__ __forceinline__ bool start_path(const DevScene& S, const Stream& A, const Pool& P, uint32_t slot) {
    while (true) {
        unsigned long long g = atomicAdd(&P.ctr[0], 1ull);
        if (g >= A.total) return false;
        int px, py;
        Rng rng;
        rng.k0 = A.k0;
        rng.k1 = A.k1;
        if (!decode_sample(A, g, px, py, rng.pixel, rng.sample)) continue;
        Ray ray = camera_ray(S, px, py, rng);
        P.ray_o[slot] = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.time);
        P.ray_d[slot] = make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(PRIM_NONE));
        P.thr[slot] = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(0u));
        P.rad[slot] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        P.id[slot] = make_uint2(rng.pixel, rng.sample);
        return true;
    }
}

// warp-aggregated append to the next active list
__device__ __forceinline__ void append_next(const Pool& P, uint32_t* next_list, bool want, uint32_t slot) {
    __syncwarp();
    const unsigned mask = __ballot_sync(0xffffffffu, want);
    if (!want) return;
    const unsigned lane = threadIdx.x & 31u;
    const int leader = __ffs(mask) - 1;
    unsigned long long base = 0;
    if ((int)lane == leader) base = atomicAdd(&P.ctr[3], (unsigned long long)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    next_list[base + __popc(mask & ((1u << lane) - 1u))] = slot;
}

__global__ void wf_generate(const __grid_constant__ DevScene S, const __grid_constant__ Stream A, const __grid_constant__ Pool P) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = false;
    if (slot < P.capacity && A.max_depth > 0) ok = start_path(S, A, P, slot);
    // generate fills list[1] as "next"; the first wf_swap makes it current
    append_next(P, P.list[1], ok, slot);
}

__global__ void wf_swap(const __grid_constant__ Pool P) {
    P.ctr[2] = P.ctr[3];
    P.ctr[3] = 0;
    P.ctr[4] = 0;
    P.ctr[5] ^= 1ull;
}

#ifndef RT_WF_REFILL
#define RT_WF_REFILL 8
#endif

template <bool STATS>
__global__ void __launch_bounds__(256, 4) wf_extend(const __grid_constant__ DevScene S, const __grid_constant__ Pool P,
                                                    Stats* __restrict__ gstats) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned n = (unsigned)P.ctr[2];
    const uint32_t* list = P.list[P.ctr[5] & 1ull];
    Stats st;
    if (STATS) memset(&st, 0, sizeof st);
    bool queue_empty = n == 0;
    bool active = false;
    uint32_t slot = 0, origin_prim = PRIM_NONE;
    Ray ray;
    ray.o = ray.d = v3(0, 0, 0);
    ray.time = 0;
    RayConst rc;
    rc.set(ray);
    Trav tr;
    StackEntry stack[STACK_SIZE];
    tr.init(S, 0.0f);
    tr.cur = LINK_DONE;

    while (true) {
        // ---- refill idle lanes from the active list ------------------------------------------
        unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (idle && !queue_empty) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&P.ctr[4], (unsigned long long)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base + __popc(idle) >= n) queue_empty = true;
            const unsigned long long e = base + __popc(idle & lt_mask);
            if (!active && e < n) {
                slot = list[e];
                const float4 o = P.ray_o[slot], d = P.ray_d[slot];
                ray.o = v3(o); ray.time = o.w;
                ray.d = v3(d); origin_prim = __float_as_uint(d.w);
                rc.set(ray);
                tr.init(S, __int_as_float(0x7f800000));
                active = true;
                if (STATS) st.rays++;
                if (tr.done()) {
                    P.hit[slot] = make_float4(tr.hit.t, __uint_as_float(tr.hit.prim), 0.0f, 0.0f);
                    active = false;
                }
            }
        }
        if (__ballot_sync(0xffffffffu, active) == 0u) {
            if (queue_empty) break;
            continue;
        }
        // ---- traverse until enough lanes are idle to make a refill worthwhile ----------------------
        while (true) {
            while (true) {
                const bool descending = active && tr.cur >= 0;
                if (__ballot_sync(0xffffffffu, descending) == 0u) break;
                if (descending) tr.interior<STATS>(S, rc, 0.001f, stack, &st);
            }
            if (active) {
                if (!tr.done()) tr.leaf<STATS>(S, ray, rc, 0.001f, origin_prim, stack, &st);
                if (tr.done()) {
                    P.hit[slot] = make_float4(tr.hit.t, __uint_as_float(tr.hit.prim), tr.hit.u, tr.hit.v);
                    active = false;
                }
            }
            const unsigned act = __ballot_sync(0xffffffffu, active);
            if (act == 0u) break;
            if (!queue_empty && 32 - __popc(act) >= RT_WF_REFILL) break;
        }
    }
    if (STATS) {
        unsigned long long* g = reinterpret_cast<unsigned long long*>(gstats);
        const unsigned long long* l = reinterpret_cast<const unsigned long long*>(&st);
        for (unsigned i = 0; i < sizeof(Stats) / 8; i++) {
            unsigned long long v = l[i];
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if (lane == 0 && v) atomicAdd(g + i, v);
        }
    }
}

template <bool STATS>
__global__ void __launch_bounds__(256, 3) wf_shade(const __grid_constant__ DevScene S, const __grid_constant__ Stream A,
                                                   const __grid_constant__ Pool P, unsigned long long* __restrict__ accum,
                                                   Stats* __restrict__ gstats) {
    const unsigned n = (unsigned)P.ctr[2];
    const unsigned cur = (unsigned)(P.ctr[5] & 1ull);
    const uint32_t* list = P.list[cur];
    uint32_t* next_list = P.list[cur ^ 1u];
    Stats st;
    if (STATS) memset(&st, 0, sizeof st);
    const unsigned stride = gridDim.x * blockDim.x;
    // every lane of a warp runs the same number of iterations (append_next uses warp votes)
    const unsigned rounds = (n + stride - 1) / stride;
    for (unsigned it = 0; it < rounds; it++) {
        const unsigned e = it * stride + blockIdx.x * blockDim.x + threadIdx.x;
        bool cont = false;
        uint32_t slot = 0;
        if (e < n) {
            slot = list[e];
            const float4 o = P.ray_o[slot], d = P.ray_d[slot], th = P.thr[slot], ra = P.rad[slot], h = P.hit[slot];
            const uint2 id = P.id[slot];
            Ray ray;
            ray.o = v3(o); ray.time = o.w; ray.d = v3(d);
            V3 T = v3(th), L = v3(ra);
            uint32_t bounce = __float_as_uint(th.w);
            Rng rng;
            rng.pixel = id.x; rng.sample = id.y; rng.k0 = A.k0; rng.k1 = A.k1;
            Hit hit;
            hit.t = h.x; hit.prim = __float_as_uint(h.y); hit.u = h.z; hit.v = h.w;
            uint32_t origin_prim = PRIM_NONE;

            // Camera.txt:203-238, one level
            int medium = -1;
            if (S.n_media > 0) medium = media_hit<STATS>(S, ray, 0.001f, hit.t, rng, bounce, &st);
            bool done = false;
            if (medium < 0 && hit.prim == PRIM_NONE) {
                L = L + T * v3(S.background);
                done = true;
            } else {
                Surface sf;
                if (medium >= 0) {  // constant_medium.h:45-50
                    const DevMedium& md = S.media[medium];
                    sf.t = hit.t;
                    sf.p = fma3(hit.t, ray.d, ray.o);
                    sf.normal = v3(md.normal);
                    sf.front = true;
                    sf.u = sf.v = 0.0f;
                    sf.material = md.material;
                    sf.prim_id = -1;
                } else {
                    complete_hit(S, ray, hit, sf, false);
                    origin_prim = hit.prim;
                }
                const DevMaterial& m = S.mats[sf.material];
                float4 u4 = make_float4(0, 0, 0, 0);
                if (m.type != RT_MAT_DIFFUSE_LIGHT && m.type != RT_MAT_EMISSIVE_LIGHT) u4 = rng.draw(bounce, RS_SCATTER);
                V3 att, emitted;
                Ray next;
                const bool scattered = shade_surface(S, m, ray, sf, [&] { return u4; }, emitted, att, next);
                L = L + T * emitted;
                if (!scattered) {
                    done = true;
                } else {
                    if (S.n_lights > 0) L = L + T * att * point_lighting(S, sf.p, sf.normal);
                    T = T * att;
                    ray = next;
                    bounce++;
                    if (bounce >= (uint32_t)A.max_depth) done = true;
                }
            }
            if (done) {
                unsigned long long* a = accum + 4ull * id.x;
                if (isfinite(L.x) && isfinite(L.y) && isfinite(L.z)) {
                    atomicAdd(a + 0, __float2ull_rn(fminf(fmaxf(L.x, 0.0f), 1048576.0f) * 268435456.0f));
                    atomicAdd(a + 1, __float2ull_rn(fminf(fmaxf(L.y, 0.0f), 1048576.0f) * 268435456.0f));
                    atomicAdd(a + 2, __float2ull_rn(fminf(fmaxf(L.z, 0.0f), 1048576.0f) * 268435456.0f));
                } else {
                    atomicAdd(a + 3, 1ull);
                    if (STATS) st.nonfinite++;
                }
                cont = start_path(S, A, P, slot);  // the slot takes the next sample of the stream
                if (STATS && cont) st.samples++;
            } else {
                P.ray_o[slot] = make_float4(ray.o.x, ray.o.y, ray.o.z, ray.time);
                P.ray_d[slot] = make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(origin_prim));
                P.thr[slot] = make_float4(T.x, T.y, T.z, __uint_as_float(bounce));
                P.rad[slot] = make_float4(L.x, L.y, L.z, 0.0f);
                cont = true;
            }
        }
        append_next(P, next_list, cont, slot);
    }
    if (STATS) {
        const unsigned lane = threadIdx.x & 31u;
        unsigned long long* g = reinterpret_cast<unsigned long long*>(gstats);
        const unsigned long long* l = reinterpret_cast<const unsigned long long*>(&st);
        for (unsigned i = 0; i < sizeof(Stats) / 8; i++) {
            unsigned long long v = l[i];
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if (lane == 0 && v) atomicAdd(g + i, v);
        }
    }
}

}  // namespace rtwf
