// rt_kernel_v3.cuh — render_kernel_v3: the v2 megakernel with TWO path contexts per lane.
//
// Measured on v2 (profiles/r1_bench_n1.json, key `lane_occupancy`): a BVH node step runs with 12 of 32
// lanes working — 13 hold a leaf and wait for the others to arrive, 7 have finished their ray and
// wait for the phase to end.  v3 gives every lane a second path: one context lives in registers
// (as in v2), the other is PARKED in shared memory (23 words per lane, field-major so that a
// warp's accesses are conflict-free).  A lane whose ray finishes swaps contexts and keeps
// traversing; the shade phase runs two rounds back to back (better instruction-cache reuse), both
// nearly full.  Because lanes are no longer in step, the node loop does not wait for ALL lanes to
// reach a leaf: it yields to the leaf code as soon as kLeafTrigger lanes hold one.
//
// Invariant: at most one context of a lane owns traversal-stack content (the stack is a per-lane
// local array).  A parked context is therefore either not traversing or FRESH (sp == 0, nothing
// visited); the only exception is transient, inside the shade phase, where a suspended traversal
// is parked while its lane shades the other path (shading does not touch the stack) and is
// swapped back before the next traversal phase.
//
// Images are bit-identical to v2's: a sample is a pure function of its Philox counter and the
// frame is a sum of integers.
#pragma once

#ifndef RT_V3_LEAF_TRIGGER
#define RT_V3_LEAF_TRIGGER 12
#endif
#ifndef RT_V3_THRESHOLD
#define RT_V3_THRESHOLD 8
#endif
#ifndef RT_V3_TAKE_MIN
#define RT_V3_TAKE_MIN 1
#endif
constexpr int kLeafTrigger = RT_V3_LEAF_TRIGGER;
constexpr int kV3Threshold = RT_V3_THRESHOLD;
constexpr int kTakeMin = RT_V3_TAKE_MIN;  // lanes that must be waiting for their parked path before the warp runs the swap code
constexpr int kParkWords = 23;

struct PathCtx {  // everything that defines a path between two steps of its state machine
    int state;
    uint32_t pixel, sample, bounce, origin_prim;
    Ray ray;
    V3 L, T;
    Hit hit;
    int cur, sp;
};

// exchange the register context with the parked one (slot = this lane's column)
__device__ __forceinline__ void swap_ctx(uint32_t* park, PathCtx& c) {
    auto xu = [&](int field, uint32_t& v) {
        uint32_t* p = park + field * 32;
        const uint32_t t = *p;
        *p = v;
        v = t;
    };
    auto xf = [&](int field, float& v) {
        uint32_t u = __float_as_uint(v);
        xu(field, u);
        v = __uint_as_float(u);
    };
    auto xi = [&](int field, int& v) {
        uint32_t u = (uint32_t)v;
        xu(field, u);
        v = (int)u;
    };
    xi(0, c.state);
    xu(1, c.pixel); xu(2, c.sample); xu(3, c.bounce); xu(4, c.origin_prim);
    xf(5, c.ray.o.x); xf(6, c.ray.o.y); xf(7, c.ray.o.z);
    xf(8, c.ray.d.x); xf(9, c.ray.d.y); xf(10, c.ray.d.z); xf(11, c.ray.time);
    xf(12, c.L.x); xf(13, c.L.y); xf(14, c.L.z);
    xf(15, c.T.x); xf(16, c.T.y); xf(17, c.T.z);
    xf(18, c.hit.t); xu(19, c.hit.prim); xf(20, c.hit.u); xf(21, c.hit.v);
    // cur and sp share a word: |cur| < 2^31 needs all 32 bits, so sp rides with the state word's
    // upper bits instead (state < 4, sp < 64)
    uint32_t packed = (uint32_t)c.cur;
    xu(22, packed);
    c.cur = (int)packed;
}

template <bool STATS, bool LITE>
__global__ void __launch_bounds__(256, RT_MIN_BLOCKS) render_kernel_v3(const __grid_constant__ DevScene S, const __grid_constant__ RenderArgs A,
                                                                       unsigned long long* __restrict__ accum,
                                                                       unsigned long long* __restrict__ counters, Stats* __restrict__ gstats) {
    __shared__ uint32_t park_all[8][kParkWords][32];
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    uint32_t* const park = &park_all[threadIdx.x >> 5][0][lane];
    Stats st;
    if (STATS) memset(&st, 0, sizeof st);

    // warp-uniform pool of (pixel, sample) pairs
    unsigned pool_pos = 0, pool_size = 0;
    int blk_x0 = 0, blk_y0 = 0, seg_s0 = 0;
    bool exhausted = A.max_depth <= 0;  // ray_color(depth <= 0) is black before anything is traced

    PathCtx c;
    c.state = LANE_IDLE;
    c.pixel = c.sample = c.bounce = 0;
    c.origin_prim = PRIM_NONE;
    c.ray.o = c.ray.d = v3(0, 0, 0);
    c.ray.time = 0;
    c.L = v3(0, 0, 0);
    c.T = v3(1, 1, 1);
    c.hit.t = 0;
    c.hit.prim = PRIM_NONE;
    c.hit.u = c.hit.v = 0;
    c.cur = LINK_DONE;
    c.sp = 0;
    // the parked context starts idle; its state is mirrored in a register
    for (int f = 0; f < kParkWords; f++) park[f * 32] = 0u;
    park[22 * 32] = (uint32_t)LINK_DONE;
    int parked_state = LANE_IDLE;
    Rng rng;
    rng.k0 = A.k0;
    rng.k1 = A.k1;
    StackEntry stack[STACK_SIZE];
    const float kInf = __int_as_float(0x7f800000);
    __syncwarp();

    // sp travels in the upper bits of the state word (see swap_ctx)
    auto do_swap = [&]() {
        c.state |= c.sp << 8;
        swap_ctx(park, c);
        c.sp = c.state >> 8;
        c.state &= 0xff;
    };

    while (true) {
        // ---- 1. shade / regenerate, two rounds: the register context, then the parked one ----------
#pragma unroll 1
        for (int round = 0; round < 2; round++) {
            bool swapped = false, started = false;
            if (round == 1) {
                // the parked path needs service: it finished its traversal, or it is idle and there
                // are samples left to start
                swapped = parked_state == LANE_SHADE || (parked_state == LANE_IDLE && !exhausted);
                if (__ballot_sync(0xffffffffu, swapped) == 0u) break;
                if (swapped) {
                    const int mine = c.state;
                    // a traversal that has taken at least one step owns the lane's stack
                    started = mine == LANE_TRAVERSE && !(c.cur == S.root && c.sp == 0);
                    do_swap();
                    parked_state = mine;
                }
            }
            // ---- shade: Camera.txt:203-238 for the lanes whose traversal finished ------------------
            if (STATS) {
                const unsigned smask = __ballot_sync(0xffffffffu, c.state == LANE_SHADE);
                if (lane == 0 && smask) { st.shade_iters++; st.shade_lanes += __popc(smask); }
            }
            if (c.state == LANE_SHADE) {
                rng.pixel = c.pixel;
                rng.sample = c.sample;
                Hit hit = c.hit;
                int medium = -1;
                if (S.n_media > 0) medium = media_hit<STATS>(S, c.ray, 0.001f, hit.t, rng, c.bounce, &st);
                bool done = false;
                if (medium < 0 && hit.prim == PRIM_NONE) {
                    c.L = c.L + c.T * v3(S.background);
                    done = true;
                } else {
                    Surface sf;
                    if (medium >= 0) {  // constant_medium.h:45-50
                        const DevMedium& md = S.media[medium];
                        sf.t = hit.t;
                        sf.p = fma3(hit.t, c.ray.d, c.ray.o);
                        sf.normal = v3(md.normal);
                        sf.front = true;
                        sf.u = sf.v = 0.0f;
                        sf.material = md.material;
                        sf.prim_id = -1;
                        c.origin_prim = PRIM_NONE;
                    } else {
                        complete_hit(S, c.ray, hit, sf, false);
                        c.origin_prim = hit.prim;
                    }
                    const DevMaterial& m = S.mats[sf.material];
                    float4 u4 = make_float4(0, 0, 0, 0);
                    if (m.type != RT_MAT_DIFFUSE_LIGHT && m.type != RT_MAT_EMISSIVE_LIGHT) u4 = rng.draw(c.bounce, RS_SCATTER);
                    V3 att, emitted;
                    Ray next;
                    const bool scattered = shade_surface(S, m, c.ray, sf, [&] { return u4; }, emitted, att, next);
                    c.L = c.L + c.T * emitted;
                    if (!scattered) {
                        done = true;
                    } else {
                        if (!LITE && S.n_lights > 0) c.L = c.L + c.T * att * point_lighting(S, sf.p, sf.normal);
                        c.T = c.T * att;
                        c.ray = next;
                        c.bounce++;
                        if (c.bounce >= (uint32_t)A.max_depth) done = true;  // ray_color(depth <= 0) returns 0
                    }
                }
                if (done) {
                    unsigned long long* a = accum + 4ull * c.pixel;
                    if (isfinite(c.L.x) && isfinite(c.L.y) && isfinite(c.L.z)) {
                        atomicAdd(a + 0, __float2ull_rn(fminf(fmaxf(c.L.x, 0.0f), kSampleClamp) * kAccumScale));
                        atomicAdd(a + 1, __float2ull_rn(fminf(fmaxf(c.L.y, 0.0f), kSampleClamp) * kAccumScale));
                        atomicAdd(a + 2, __float2ull_rn(fminf(fmaxf(c.L.z, 0.0f), kSampleClamp) * kAccumScale));
                    } else {
                        atomicAdd(a + 3, 1ull);
                        if (STATS) st.nonfinite++;
                    }
                    c.state = LANE_IDLE;
                } else {
                    c.hit.t = kInf;
                    c.hit.prim = PRIM_NONE;
                    c.hit.u = c.hit.v = 0.0f;
                    c.sp = 0;
                    c.cur = S.n_world > 0 ? S.root : LINK_DONE;
                    c.state = c.cur == LINK_DONE ? LANE_SHADE : LANE_TRAVERSE;
                    if (STATS) st.rays++;
                }
            }
            // ---- regenerate: idle lanes take the next (pixel, sample) pairs of the pool ------------
            unsigned needy = __ballot_sync(0xffffffffu, c.state == LANE_IDLE);
            while (needy && !exhausted) {
                if (pool_pos >= pool_size) {
                    unsigned long long item = 0;
                    if (lane == 0) item = atomicAdd(&counters[0], 1ull);
                    item = __shfl_sync(0xffffffffu, item, 0);
                    if (item >= A.n_items) {
                        exhausted = true;
                        break;
                    }
                    const unsigned seg = (unsigned)(item % (unsigned long long)A.n_segments);
                    const unsigned long long blk = item / (unsigned long long)A.n_segments;
                    const unsigned blocks_per_tile = (unsigned)(A.blocks_per_tile_x * A.blocks_per_tile_y);
                    const unsigned local_tile = (unsigned)(blk / blocks_per_tile), in_tile = (unsigned)(blk % blocks_per_tile);
                    const unsigned tile = A.tile_offset + local_tile * A.tile_stride;
                    blk_x0 = (int)(tile % A.tiles_x) * A.tile_size + (int)(in_tile % A.blocks_per_tile_x) * 8;
                    blk_y0 = (int)(tile / A.tiles_x) * A.tile_size + (int)(in_tile / A.blocks_per_tile_x) * 4;
                    seg_s0 = (int)seg * A.seg_len;
                    pool_size = 32u * (unsigned)min(A.seg_len, A.n_local_samples - seg_s0);
                    pool_pos = 0;
                }
                const unsigned e = pool_pos + __popc(needy & lt_mask);
                if (c.state == LANE_IDLE && e < pool_size) {
                    const int px = blk_x0 + (int)(e & 7u), py = blk_y0 + (int)((e >> 3) & 3u);
                    if (px < A.width && py < A.height) {
                        c.pixel = rng.pixel = (uint32_t)(py * A.width + px);
                        c.sample = rng.sample = (uint32_t)(A.spp_begin + A.sample_offset + (seg_s0 + (int)(e >> 5)) * A.sample_stride);
                        c.ray = camera_ray<LITE>(S, px, py, rng);
                        c.L = v3(0, 0, 0);
                        c.T = v3(1, 1, 1);
                        c.bounce = 0;
                        c.origin_prim = PRIM_NONE;
                        c.hit.t = kInf;
                        c.hit.prim = PRIM_NONE;
                        c.hit.u = c.hit.v = 0.0f;
                        c.sp = 0;
                        c.cur = S.n_world > 0 ? S.root : LINK_DONE;
                        c.state = c.cur == LINK_DONE ? LANE_SHADE : LANE_TRAVERSE;
                        if (STATS) { st.samples++; st.rays++; }
                    }
                }
                pool_pos += min((unsigned)__popc(needy), pool_size - pool_pos);
                needy = __ballot_sync(0xffffffffu, c.state == LANE_IDLE);
            }
            // a suspended traversal that was parked for this round comes back to the registers (it
            // owns the stack); a fresh one may stay parked
            if (round == 1 && started) {
                const int mine = c.state;
                do_swap();
                parked_state = mine;
            }
        }
        // a lane whose register path has nothing to traverse but whose parked one has: swap
        if (c.state != LANE_TRAVERSE && parked_state == LANE_TRAVERSE) {
            const int mine = c.state;
            do_swap();
            parked_state = mine;
        }
        const unsigned busy = __ballot_sync(0xffffffffu, c.state != LANE_IDLE || parked_state != LANE_IDLE);
        if (busy == 0u) break;  // pool dry, nothing in flight
        if (__ballot_sync(0xffffffffu, c.state == LANE_TRAVERSE) == 0u) continue;  // only world-less shading left

        // ---- 2. traversal phase ------------------------------------------------------------------
        {
            RayConst rc;
            rc.set(c.ray);
            Trav tr;
            tr.hit = c.hit;
            tr.cur = c.cur;
            tr.sp = c.sp;
            while (true) {
                // descend: lanes holding an interior node step; lanes holding a leaf wait, but only
                // until kLeafTrigger of them do
                while (true) {
                    const bool descending = c.state == LANE_TRAVERSE && tr.cur >= 0;
                    const unsigned dmask = __ballot_sync(0xffffffffu, descending);
                    if (dmask == 0u) break;
                    const unsigned lmask = __ballot_sync(0xffffffffu, c.state == LANE_TRAVERSE && tr.cur < 0);
                    if (__popc(lmask) >= kLeafTrigger) break;
                    if (STATS && lane == 0) { st.desc_iters++; st.desc_lanes += __popc(dmask); st.desc_trav_lanes += __popc(dmask | lmask); }
                    if (descending) tr.interior<STATS>(S, rc, 0.001f, stack, &st);
                }
                if (STATS) {
                    const unsigned lm = __ballot_sync(0xffffffffu, c.state == LANE_TRAVERSE && tr.cur < 0 && !tr.done());
                    if (lane == 0 && lm) { st.leaf_iters++; st.leaf_lanes += __popc(lm); }
                }
                if (c.state == LANE_TRAVERSE && tr.cur < 0) {
                    if (!tr.done()) tr.leaf<STATS, LITE>(S, c.ray, rc, 0.001f, c.origin_prim, stack, &st);
                    if (tr.done()) c.state = LANE_SHADE;
                }
                // a lane whose ray is finished continues with its parked path, if that one is waiting
                // to be traced
                const bool take = c.state == LANE_SHADE && parked_state == LANE_TRAVERSE;
                if (__popc(__ballot_sync(0xffffffffu, take)) >= kTakeMin) {
                    if (take) {
                        c.hit = tr.hit;
                        c.cur = tr.cur;
                        c.sp = 0;
                        do_swap();
                        parked_state = LANE_SHADE;
                        rc.set(c.ray);
                        tr.hit = c.hit;
                        tr.cur = c.cur;
                        tr.sp = c.sp;
                    }
                }
                const unsigned active = __ballot_sync(0xffffffffu, c.state == LANE_TRAVERSE);
                if (active == 0u || __popc(active) < kV3Threshold) break;
            }
            c.hit = tr.hit;
            c.cur = tr.cur;
            c.sp = tr.sp;
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
