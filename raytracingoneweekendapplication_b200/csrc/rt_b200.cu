// rt_b200.cu — the C ABI of include/rt_b200.h: scene upload (flatten -> bake -> SAH BVH ->
// device layout) and the sm_100a kernels of the path-tracing hot path.
//
// Kernel inventory (hand-written; the device builder of bvh_device.cuh also runs cub's sort and scan):
//   render_kernel_v2<STATS, LITE, NEE, WIDTH, FEAT, MOMENTS, VIEWS>
//                          the persistent megakernel that renders: raygen -> traverse -> media ->
//                          shade -> accumulate, per-warp streams of (pixel, sample) pairs and 64-bit
//                          fixed-point accumulation.  Its compiled instances are the rows of kV2Instances
//   aov_kernel             deterministic primary hits (parity tests)
//   resolve_kernel         accumulation buffer -> float radiance + RGB8 (Camera.txt:74-89)
//   variance_kernel, noise_kernel   sums + second moments -> per-pixel sample variance, frame noise partials
//   untile_kernel, add_sums_kernel   shard frames: compact tiles -> full frame, sums
//   pair_nodes_kernel      device-built BVH2 nodes -> the paired layout the traversal reads
//   probe_*_kernel         per-function known-answer probes
//   fma_peak_kernel, l1_peak_kernel   FP32 and L1 roofline denominators
//   rtlbvh::*              the device BVH builder (bvh_device.cuh)
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "bvh_build.h"
#include "bvh_wide.h"
#include "prim_derive.h"
#include "bvh_device.cuh"
#include "rt_b200.h"
#include "rt_device.cuh"
#include "rt_wide.cuh"

using namespace rtdev;

// ---------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------
struct RenderArgs {
    int width, height;
    int max_depth;
    int spp_begin;       // first sample index of this call
    int n_local_samples; // samples this shard traces per pixel
    int sample_stride, sample_offset;  // global sample = spp_begin + sample_offset + k * sample_stride
    int seg_len;         // samples per work item
    int n_segments;
    int tiles_x, tiles_y, tile_size;
    int tile_stride, tile_offset;      // global tile = tile_offset + k * tile_stride
    int n_local_tiles;
    int blocks_per_tile_x, blocks_per_tile_y;  // 8x4 pixel blocks per tile
    uint32_t side_lo;        // the side pointer, its two 32-bit halves in the struct's two alignment holes (here and after
                             // shadow_point_lights), so that no offset of a field or a kernel parameter moves.  It serves the
                             // instances that need it, which are never the same: MOMENTS, the moments buffer (unsigned long
                             // long); VIEWS, the view table (ViewRecord)
    unsigned long long n_items;
    uint32_t k0, k1;
    int compact;             // RT_FLAG_COMPACT_TILES: `accum` holds only this shard's tiles, tile-major: slot = local_tile * tile_size^2 + y_in_tile * tile_size + x_in_tile
    int nee_emitters;        // NEE instance: sample the listed quad emitters (RT_FLAG_NEE)
    int shadow_point_lights; // NEE instance: shadow rays for the point lights (RT_FLAG_SHADOWED_POINT_LIGHTS)
    uint32_t side_hi;
    template <class T>
    __host__ __device__ T* side() const { return (T*)(((uint64_t)side_hi << 32) | side_lo); }
    void set_side(const void* p) { side_lo = (uint32_t)(uintptr_t)p; side_hi = (uint32_t)((uint64_t)(uintptr_t)p >> 32); }
};
static_assert(sizeof(RenderArgs) == 104 && offsetof(RenderArgs, n_items) == 72, "the side pointer fills alignment holes only");

constexpr float kAccumScale = 268435456.0f;  // 2^RT_ACCUM_FRAC_BITS
constexpr float kSampleClamp = 1048576.0f;   // 2^20: keeps 2^16 saturated samples inside 64 bits

// RT_FLAG_MOMENTS: the second moment of a sample.  x is the exact integer added to a radiance word (x <= 2^48 after the
// clamp), so x^2 <= 2^96 is exact in 128 bits; it is added as two 48-bit limbs, m[0] += x^2 mod 2^48 and
// m[1] += x^2 >> 48, each < 2^48 except m[1] = 2^48 for a sample saturated at kSampleClamp.  With at most 2^16 samples
// per pixel a limb word stays below 2^64 however the samples are split -- save for 2^16 samples that ALL saturate,
// the edge the radiance words share (kSampleClamp).  A zero limb (every black sample) costs no atomic.
__device__ __forceinline__ void add_square(unsigned long long* m, unsigned long long x) {
    const unsigned long long lo = x * x, hi = __umul64hi(x, x);
    const unsigned long long l0 = lo & ((1ull << 48) - 1ull), l1 = (lo >> 48) | (hi << 16);
    if (l0) atomicAdd(m, l0);
    if (l1) atomicAdd(m + 1, l1);
}

// ---------------------------------------------------------------------------------
// render_kernel_v2 — the production megakernel.
//
// ncu on the first version (profiles/r1_v1_*.txt) showed 7.8 of 32 threads active per issued
// instruction: (1) lanes that finished their fixed share of samples idled until the slowest
// lane of the warp was through, and (2) inside the traversal every lane waited for the
// longest ray of the warp.  v2 is organised as a per-warp STREAM instead:
//   * a warp owns no pixels.  It pulls (8x4 pixel block x sample segment) items from a global
//     counter into a pool of 32 * seg_len (pixel, sample) pairs; an idle lane takes the next
//     pair of the pool, whatever pixel it belongs to.  Radiance goes to the frame with three
//     64-bit integer REDs per finished sample, so who traced what does not matter
//     (order-independent fixed-point sums keep the image bit-identical).
//   * each lane is a small state machine: IDLE -> TRAVERSE -> SHADE -> TRAVERSE ... -> IDLE.
//     The warp alternates between a traversal phase, in which lanes step through the BVH
//     ("while-while": all lanes descend interior nodes until each holds a leaf, then all
//     intersect their leaf), and a shade phase.  The traversal phase is left as soon as fewer
//     than kTravThreshold lanes still have a ray in flight; those are suspended with their
//     stack, the others shade/regenerate, and the next traversal phase runs full again.
// ---------------------------------------------------------------------------------
#ifndef RT_TRAV_THRESHOLD
#define RT_TRAV_THRESHOLD 4
#endif
#ifndef RT_B200_DEFAULT_BVH_WIDTH
#define RT_B200_DEFAULT_BVH_WIDTH 2  // the default is decided by measurement (DESIGN.md section 3b)
#endif
#ifndef RT_MIN_BLOCKS
#define RT_MIN_BLOCKS 4  // blocks of RT_V2_THREADS per SM the binary instances are compiled for: 4 x 256 = 32 warps at 64 registers
                         // (round 1 ran 3 x 256 at 80 registers; re-measured on the round-2 kernel, profiles/r2_block_shape_sweep.txt)
#endif
#ifndef RT_WIDE_MIN_BLOCKS
#define RT_WIDE_MIN_BLOCKS RT_MIN_BLOCKS  // blocks per SM the wide instances are compiled for (register budget)
#endif
#ifndef RT_V2_THREADS
#define RT_V2_THREADS 256  // threads per block of render_kernel_v2 (tuning experiments: 224 x 3 trades warps for registers)
#endif
// STATS only: histograms of the shape of a ray's traversal, written behind the Stats block --
// node steps before the first leaf [0,64), between two leaf visits [64,128), after the last
// leaf (or of a ray that reaches none) [128,192), and leaf visits per ray [192,208)
constexpr int kTravHistBins = 208;
constexpr int kTravThreshold = RT_TRAV_THRESHOLD;
enum : int { LANE_IDLE = 0, LANE_TRAVERSE = 1, LANE_SHADE = 2 };

// WIDTH: which acceleration structure the instance traverses -- 2: the binary tree of 64-byte nodes
// (Trav, stack in local memory), 8 / 4: the wide quantised tree (TravW, rt_wide.cuh; stack in dynamic
// shared memory, [entry][thread], `A.stack_entries` entries per thread)
template <int WIDTH>
struct TravSel { using Trav = TravW<WIDTH>; using RayConst = RayConstW; };
template <>
struct TravSel<2> { using Trav = rtdev::Trav; using RayConst = rtdev::RayConst; };

// FEAT: which rarely needed code the instance carries (like LITE: code that never runs still costs registers and spills).
//   FEAT_MEDIA          the scene has a constant_medium (without: C1, C2, C4 -- +2 %, +1.9 %, +3.4 %)
//   FEAT_MEDIA_GENERAL  some boundary is not one static sphere (C3's boxes; without: C5 +3.7 %)
//   FEAT_SPECULAR       some material is RT_MAT_SPECULAR (without: C5 +0.6 %)
//   FEAT_MSPHERE        the world holds a moving sphere (C5 has one)
//   FEAT_TRI / FEAT_LIGHTS / FEAT_DEFOCUS   triangles / point lights / defocus blur: what LITE = true removes together;
//                       a LITE = false instance carries only those of the three its mask names (C1: defocus only,
//                       C4: triangles and point lights)
// The plain binary-tree kernel is compiled for the masks listed in kV2Instances; a scene runs the first one that covers it.
enum : int { FEAT_MEDIA = 1, FEAT_MEDIA_GENERAL = 2, FEAT_SPECULAR = 4, FEAT_MSPHERE = 8, FEAT_TRI = 16, FEAT_LIGHTS = 32,
             FEAT_DEFOCUS = 64, FEAT_ALL = 127 };
// One 16-byte slot of local memory per lane, moved with one vector store and one vector load.  The accesses are
// volatile PTX, so the value stays in the slot between them instead of occupying registers or scattered scalar spills.
struct LocalSlot {
    float4 mem;
    __device__ __forceinline__ void store(float4 v) {
        asm volatile("st.local.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(__cvta_generic_to_local(&mem)), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
    }
    __device__ __forceinline__ float4 load() {
        float4 v;
        asm volatile("ld.local.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(__cvta_generic_to_local(&mem)));
        return v;
    }
};

// MOMENTS: also add the second moments of every finished sample to A.side() (6 words per slot, see add_square)
// VIEWS: a multi-view batch (rt_render_views).  The local tiles run over views x tiles of one view's frame, view-major
// (item / items_per_view = tile / (tiles_x * tiles_y) is the view); each lane takes camera and Philox key from its view's
// record in A.side() and accumulates into slot view * width * height + pixel of `accum`, kept in lane_slot like a
// compact tile slot.  Never with STATS, MOMENTS, compact tiles or shards.
template <bool STATS, bool LITE, bool NEE = false, int WIDTH = 2, int FEAT = FEAT_ALL, bool MOMENTS = false, bool VIEWS = false>
__global__ void __launch_bounds__(RT_V2_THREADS, WIDTH == 2 ? RT_MIN_BLOCKS : RT_WIDE_MIN_BLOCKS) render_kernel_v2(const __grid_constant__ DevScene S, const __grid_constant__ RenderArgs A,
                                                        unsigned long long* __restrict__ accum,
                                                        unsigned long long* __restrict__ counters, Stats* __restrict__ gstats) {
    constexpr bool NO_TRI = LITE || !(FEAT & FEAT_TRI), NO_DEFOCUS = LITE || !(FEAT & FEAT_DEFOCUS), LIGHTS = !LITE && (FEAT & FEAT_LIGHTS);
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    Stats st;
    if (STATS) memset(&st, 0, sizeof st);

    // warp-uniform pool of (pixel, sample) pairs
    unsigned pool_pos = 0, pool_size = 0;
    int blk_x0 = 0, blk_y0 = 0, seg_s0 = 0;
    // compact tile buffers: where a lane's current sample goes.  One word of shared memory per lane, written
    // when the sample starts and read when it ends -- no register is held across the whole path for it
    __shared__ uint32_t lane_slot[RT_V2_THREADS];
    unsigned slot_base = 0;  // compact tiles: the slot of the pool's pixel block; VIEWS (never compact): the pool's view
    bool exhausted = A.max_depth <= 0;  // ray_color(depth <= 0) is black before anything is traced

    int state = LANE_IDLE;
    Rng rng;
    rng.pixel = rng.sample = 0;
    rng.k0 = A.k0;
    rng.k1 = A.k1;
    Ray ray;
    ray.o = ray.d = v3(0, 0, 0);
    ray.time = 0;
    // the path's radiance L and throughput T live in local memory between shade phases: written where a sample starts
    // and at the end of each shade phase, read once in the shade phase, after the surface has been shaded.  Held in
    // registers, they were spilled by the compiler around the traversal phase and the out-of-line calls of the shade phase.
    LocalSlot radiance, throughput;
    uint32_t bounce = 0, origin_prim = PRIM_NONE;
    float nee_pdf = 0.0f;  // NEE: > 0 when the previous vertex sampled the listed emitters directly: the density of the direction it scattered into
    typename TravSel<WIDTH>::Trav tr;
    StackEntry stack_mem[WIDTH == 2 ? STACK_SIZE : 1];
    extern __shared__ uint2 wide_stack_mem[];
    auto stack = [&]() {
        if constexpr (WIDTH == 2) return &stack_mem[0];
        else return SmemStack<RT_V2_THREADS>::make(wide_stack_mem);
    }();
    tr.clear();
    tr.hit.t = 0;
    tr.hit.prim = PRIM_NONE;
    tr.hit.u = tr.hit.v = 0;
    const float kInf = __int_as_float(0x7f800000);
    unsigned seg_steps = 0, n_leaf = 0;  // STATS: shape of the current ray's traversal
    unsigned long long* hist = reinterpret_cast<unsigned long long*>(gstats + 1);

    while (true) {
        // ---- 1. idle lanes take the next (pixel, sample) pairs of the pool -----------------------
        unsigned needy = __ballot_sync(0xffffffffu, state == LANE_IDLE);
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
                unsigned tile = A.tile_offset + local_tile * A.tile_stride;
                if constexpr (VIEWS) {
                    const unsigned tiles_per_view = (unsigned)(A.tiles_x * A.tiles_y);
                    slot_base = tile / tiles_per_view;
                    tile -= slot_base * tiles_per_view;
                }
                blk_x0 = (int)(tile % A.tiles_x) * A.tile_size + (int)(in_tile % A.blocks_per_tile_x) * 8;
                blk_y0 = (int)(tile / A.tiles_x) * A.tile_size + (int)(in_tile / A.blocks_per_tile_x) * 4;
                seg_s0 = (int)seg * A.seg_len;
                pool_size = 32u * (unsigned)min(A.seg_len, A.n_local_samples - seg_s0);
                pool_pos = 0;
                if constexpr (!VIEWS)
                    slot_base = (local_tile * (unsigned)A.tile_size + (in_tile / (unsigned)A.blocks_per_tile_x) * 4u) * (unsigned)A.tile_size +
                                (in_tile % (unsigned)A.blocks_per_tile_x) * 8u;
            }
            const unsigned e = pool_pos + __popc(needy & lt_mask);
            if (state == LANE_IDLE && e < pool_size) {
                const int px = blk_x0 + (int)(e & 7u), py = blk_y0 + (int)((e >> 3) & 3u);
                if (px < A.width && py < A.height) {
                    rng.pixel = (uint32_t)(py * A.width + px);
                    rng.sample = (uint32_t)(A.spp_begin + A.sample_offset + (seg_s0 + (int)(e >> 5)) * A.sample_stride);
                    if (A.compact) lane_slot[threadIdx.x] = slot_base + ((e >> 3) & 3u) * (unsigned)A.tile_size + (e & 7u);
                    if constexpr (VIEWS) {
                        const ViewRecord& V = A.side<const ViewRecord>()[slot_base];
                        lane_slot[threadIdx.x] = slot_base * (unsigned)(A.width * A.height) + rng.pixel;
                        rng.k0 = V.k0;
                        rng.k1 = V.k1;
                        ray = camera_ray<NO_DEFOCUS>(V, px, py, rng);
                    } else {
                        ray = camera_ray<NO_DEFOCUS>(S, px, py, rng);
                    }
                    radiance.store(make_float4(0, 0, 0, 0));
                    throughput.store(make_float4(1, 1, 1, 0));
                    bounce = 0;
                    origin_prim = PRIM_NONE;
                    nee_pdf = 0.0f;
                    tr.init(S, kInf);
                    state = tr.done() ? LANE_SHADE : LANE_TRAVERSE;
                    if (STATS) { st.samples++; st.rays++; seg_steps = n_leaf = 0; }
                }
            }
            pool_pos += min((unsigned)__popc(needy), pool_size - pool_pos);
            needy = __ballot_sync(0xffffffffu, state == LANE_IDLE);
        }
        if (__ballot_sync(0xffffffffu, state != LANE_IDLE) == 0u) break;  // pool dry, nothing in flight

        // ---- 2. traversal phase ------------------------------------------------------------------
        {
            typename TravSel<WIDTH>::RayConst rc;
            rc.set(ray);
            while (true) {
                // descend: every traversing lane that holds an interior node takes one step per
                // iteration; lanes that reached a leaf wait until no lane of the warp descends
                while (true) {
                    // a lane that is not traversing holds LINK_DONE (negative), so the link alone says who
                    // descends; the vote goes straight to a predicate (two instructions fewer per step: +1.2 % on C5)
                    const bool descending = tr.wants_node();
                    if (!STATS) {
                        if (!__any_sync(0xffffffffu, descending)) break;
                    }
                    const unsigned dmask = STATS ? __ballot_sync(0xffffffffu, descending) : 1u;
                    if (dmask == 0u) break;
                    if (STATS) {
                        const unsigned tmask = __ballot_sync(0xffffffffu, state == LANE_TRAVERSE);
                        if (lane == 0) { st.desc_iters++; st.desc_lanes += __popc(dmask); st.desc_trav_lanes += __popc(tmask); }
                    }
                    if (descending) {
                        tr.template node_step<STATS>(S, ray, rc, 0.001f, stack, &st);
                        if (STATS) {
                            seg_steps++;
                            if (tr.done()) {
                                atomicAdd(hist + 128 + min(seg_steps, 63u), 1ull);
                                atomicAdd(hist + 192 + min(n_leaf, 15u), 1ull);
                            }
                        }
                    }
                }
                if (STATS) {
                    const unsigned lmask = __ballot_sync(0xffffffffu, state == LANE_TRAVERSE && !tr.wants_node() && !tr.done());
                    if (lane == 0 && lmask) { st.leaf_iters++; st.leaf_lanes += __popc(lmask); }
                }
                if (state == LANE_TRAVERSE && !tr.wants_node()) {
                    if (!tr.done()) {
                        tr.template leaf_step<STATS, NO_TRI, (FEAT & FEAT_MSPHERE) != 0>(S, ray, rc, 0.001f, origin_prim, stack, &st);
                        if (STATS) {
                            atomicAdd(hist + (n_leaf ? 64 : 0) + min(seg_steps, 63u), 1ull);
                            n_leaf++;
                            seg_steps = 0;
                            if (tr.done()) {
                                atomicAdd(hist + 128, 1ull);
                                atomicAdd(hist + 192 + min(n_leaf, 15u), 1ull);
                            }
                        }
                    }
                    if (tr.done()) state = LANE_SHADE;
                }
                const unsigned active = __ballot_sync(0xffffffffu, state == LANE_TRAVERSE);
                if (active == 0u || __popc(active) < kTravThreshold) break;
            }
        }

        // ---- 3. shade phase: Camera.txt:203-238 for the lanes whose traversal finished ------------
        if (STATS) {
            const unsigned smask = __ballot_sync(0xffffffffu, state == LANE_SHADE);
            if (lane == 0) { st.shade_iters++; st.shade_lanes += __popc(smask); }
        }
        if (state == LANE_SHADE) {
            V3 L, T;
            auto load_path = [&] {
                const float4 l4 = radiance.load(), t4 = throughput.load();
                L = v3(l4.x, l4.y, l4.z);
                T = v3(t4.x, t4.y, t4.z);
            };
            Hit hit = tr.hit;
            int medium = -1;
            if ((FEAT & FEAT_MEDIA) && S.n_media > 0) medium = media_hit<STATS, (FEAT & FEAT_MEDIA_GENERAL) != 0>(S, ray, 0.001f, hit.t, rng, bounce, &st);
            bool done = false;
            if (medium < 0 && hit.prim == PRIM_NONE) {
                load_path();
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
                    sf.nee_light = 0;
                    origin_prim = PRIM_NONE;
                } else {
                    complete_hit<NO_TRI, (FEAT & FEAT_MSPHERE) != 0>(S, ray, hit, sf, false);
                    origin_prim = hit.prim;
                }
                const DevMaterial& m = S.mats[sf.material];
                V3 att, emitted;
                Ray next;
                const bool scattered = shade_surface<(FEAT & FEAT_SPECULAR) != 0>(S, m, ray, sf, [&] { return rng.draw(bounce, RS_SCATTER); },
                                                                                  emitted, att, next);
                // NEE: a listed emitter reached from a vertex that also sampled the emitters directly shares the
                // estimate with that sample (balance heuristic)
                if (NEE && nee_pdf > 0.0f && medium < 0 && sf.nee_light > 0) {
                    const float d2 = dot(ray.d, ray.d);
                    const float cos_y = fabsf(dot(ray.d, v3(S.nee_lights[sf.nee_light - 1].n))) * rsqrtf(d2);
                    const float p_light = light_density(S, sf.t * sf.t * d2, fmaxf(cos_y, 1e-20f));
                    emitted = (nee_pdf / (nee_pdf + p_light)) * emitted;
                }
                load_path();
                L = L + T * emitted;
                if (!scattered) {
                    done = true;
                } else {
                    if (LIGHTS && S.n_lights > 0) {
                        if (NEE && A.shadow_point_lights) L = L + T * att * point_lighting_shadowed<WIDTH>(S, sf.p, sf.normal, origin_prim, ray.time);
                        else L = L + T * att * point_lighting(S, sf.p, sf.normal);
                    }
                    if (NEE) {
                        nee_pdf = 0.0f;
                        if (A.nee_emitters && S.n_nee_lights > 0 && (m.type == RT_MAT_LAMBERTIAN || m.type == RT_MAT_ISOTROPIC)) {
                            const bool iso = m.type == RT_MAT_ISOTROPIC;
                            nee_pdf = scatter_density(normalize(next.d), sf.normal, iso);
                            L = L + T * att * nee_direct<WIDTH>(S, sf.p, sf.normal, iso, origin_prim, ray.time, rng.draw(bounce, RS_NEE));
                        }
                    }
                    T = T * att;
                    ray = next;
                    bounce++;
                    if (bounce >= (uint32_t)A.max_depth) done = true;  // ray_color(depth <= 0) returns 0
                }
            }
            if (done) {
                unsigned long long* a = accum + 4ull * ((VIEWS || A.compact) ? lane_slot[threadIdx.x] : rng.pixel);
                if (isfinite(L.x) && isfinite(L.y) && isfinite(L.z)) {
                    atomicAdd(a + 0, __float2ull_rn(fminf(fmaxf(L.x, 0.0f), kSampleClamp) * kAccumScale));
                    atomicAdd(a + 1, __float2ull_rn(fminf(fmaxf(L.y, 0.0f), kSampleClamp) * kAccumScale));
                    atomicAdd(a + 2, __float2ull_rn(fminf(fmaxf(L.z, 0.0f), kSampleClamp) * kAccumScale));
                    if constexpr (MOMENTS) {
                        unsigned long long* m = A.side<unsigned long long>() + 6ull * (A.compact ? lane_slot[threadIdx.x] : rng.pixel);
                        add_square(m + 0, __float2ull_rn(fminf(fmaxf(L.x, 0.0f), kSampleClamp) * kAccumScale));
                        add_square(m + 2, __float2ull_rn(fminf(fmaxf(L.y, 0.0f), kSampleClamp) * kAccumScale));
                        add_square(m + 4, __float2ull_rn(fminf(fmaxf(L.z, 0.0f), kSampleClamp) * kAccumScale));
                    }
                } else {
                    atomicAdd(a + 3, 1ull);
                    if (STATS) st.nonfinite++;
                }
                state = LANE_IDLE;
                // an idle lane's traversal state is never read, but unless it is set here the previous ray's hit and
                // links stay live through the whole shade phase
                tr.init(S, kInf);
                tr.clear();
            } else {
                radiance.store(make_float4(L.x, L.y, L.z, 0.0f));
                throughput.store(make_float4(T.x, T.y, T.z, 0.0f));
                tr.init(S, kInf);
                state = tr.done() ? LANE_SHADE : LANE_TRAVERSE;
                if (STATS) { st.rays++; seg_steps = n_leaf = 0; }
            }
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

// Every compiled instance of render_kernel_v2, by its template parameters.  A request runs the first entry that covers it
// (v2_select), so the order is the preference: the per-scene feature instances of the plain binary-tree kernel (see FEAT_*
// above), then the general ones, LITE before plain.  NEE, MOMENTS and VIEWS exist for the binary tree only (every scene
// has one; shadow rays and paths then both go through it), and only as general instances.
typedef void (*RenderKernel)(const DevScene, const RenderArgs, unsigned long long*, unsigned long long*, Stats*);
struct V2Instance {
    bool stats, lite, nee, moments, views;  // lite: the scene must be LITE (no triangles, point lights, defocus)
    int width;
    int feat;  // FEAT_* bits the instance carries
    RenderKernel kernel;
};
#define RT_V2(S, L, N, M, V, W, F) {S, L, N, M, V, W, F, render_kernel_v2<S, L, N, W, F, M, V>}
static const V2Instance kV2Instances[] = {
    RT_V2(false, true, false, false, false, 2, 0),                                  // C2: quads, nothing else
    RT_V2(false, true, false, false, false, 2, FEAT_MEDIA | FEAT_MSPHERE),          // C5: media bounded by spheres, a moving sphere
    RT_V2(false, true, false, false, false, 2, FEAT_MEDIA | FEAT_MEDIA_GENERAL),    // C3: media bounded by boxes
    RT_V2(false, false, false, false, false, 2, FEAT_DEFOCUS),                      // C1: defocus blur, nothing else
    RT_V2(false, false, false, false, false, 2, FEAT_TRI | FEAT_LIGHTS),            // C4: triangles and point lights
    RT_V2(false, true, false, false, false, 2, FEAT_ALL),                           // LITE
    RT_V2(false, false, false, false, false, 2, FEAT_ALL),                          // plain
    RT_V2(true, false, false, false, false, 2, FEAT_ALL),                           // STATS
    RT_V2(false, true, false, false, false, 4, FEAT_ALL),
    RT_V2(false, false, false, false, false, 4, FEAT_ALL),
    RT_V2(true, false, false, false, false, 4, FEAT_ALL),
    RT_V2(false, true, false, false, false, 8, FEAT_ALL),
    RT_V2(false, false, false, false, false, 8, FEAT_ALL),
    RT_V2(true, false, false, false, false, 8, FEAT_ALL),
    RT_V2(false, true, true, false, false, 2, FEAT_ALL),                            // NEE + LITE
    RT_V2(false, false, true, false, false, 2, FEAT_ALL),                           // NEE
    RT_V2(false, true, false, true, false, 2, FEAT_ALL),                            // MOMENTS twins
    RT_V2(false, false, false, true, false, 2, FEAT_ALL),
    RT_V2(false, true, true, true, false, 2, FEAT_ALL),
    RT_V2(false, false, true, true, false, 2, FEAT_ALL),
    RT_V2(false, true, false, false, true, 2, FEAT_ALL),                            // VIEWS twins (rt_render_views)
    RT_V2(false, false, false, false, true, 2, FEAT_ALL),
    RT_V2(false, true, true, false, true, 2, FEAT_ALL),
    RT_V2(false, false, true, false, true, 2, FEAT_ALL),
};
#undef RT_V2

// What a pass asks of the kernel: nee = NEE or shadowed point lights; lite = the scene (and every view) allows LITE;
// width = the uploaded tree; feat = the FEAT_* bits the scene needs (FEAT_ALL: a general instance)
struct V2Key {
    bool stats, lite, nee, moments, views;
    int width;
    int feat;
};
static const V2Instance* v2_select(const V2Key& k) {
    const int width = (k.nee || k.moments || k.views) ? 2 : k.width;  // binary tree only
    for (const V2Instance& e : kV2Instances)
        if (e.stats == k.stats && e.nee == k.nee && e.moments == k.moments && e.views == k.views && e.width == width &&
            (!e.lite || k.lite) && (k.feat & ~e.feat) == 0)
            return &e;
    return nullptr;
}

// one ray through whichever acceleration structure the scene was uploaded with (test kernels)
__device__ __forceinline__ void traverse_uploaded(const DevScene& S, const Ray& ray, float tmin, float tmax, Hit& hit) {
    if (S.wide_width == 8) traverse_sel<8>(S, ray, tmin, tmax, PRIM_NONE, hit);
    else if (S.wide_width == 4) traverse_sel<4>(S, ray, tmin, tmax, PRIM_NONE, hit);
    else traverse_sel<2>(S, ray, tmin, tmax, PRIM_NONE, hit);
}

// The builders (host SAH, device LBVH + SAH top) write a node as {lmin, llink | lmax, rlink | rmin, - | rmax, -}.  The
// traversal reads the PAIRED form {lmin.x, rmin.x, lmin.y, rmin.y | lmin.z, rmin.z, lmax.x, rmax.x | lmax.y, rmax.y,
// lmax.z, rmax.z | llink, rlink, -, -}: the same plane of both children in one 64-bit register pair, which is what FFMA2
// takes (Trav::interior).  Same 64 bytes, permuted once at upload (host trees on the host, device-built trees in place).
__host__ __device__ inline void pair_node(float4* n) {
    const float4 a = n[0], b = n[1], c = n[2], e = n[3];
    n[0] = make_float4(a.x, c.x, a.y, c.y);
    n[1] = make_float4(a.z, c.z, b.x, e.x);
    n[2] = make_float4(b.y, e.y, b.z, e.z);
    n[3] = make_float4(a.w, b.w, 0.0f, 0.0f);
}
__global__ void pair_nodes_kernel(float4* __restrict__ nodes, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) pair_node(nodes + 4 * (size_t)i);
}
#include "bvh_refit.cuh"

// Camera.txt:136-168 in double: the pixel-centre ray of pixel (i, j) is center + t * (dir00 + i du + j dv)
struct CameraD {
    double center[3], dir00[3], du[3], dv[3];
};

__global__ void aov_kernel(const __grid_constant__ DevScene S, const __grid_constant__ CameraD C, int width, int height,
                           int* __restrict__ prim_id, float* __restrict__ t_out, float* __restrict__ normal, float* __restrict__ point,
                           float* __restrict__ uv) {
    int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= width || j >= height) return;
    // the ray in double (what the reference casts), rounded once for the FP32 traversal
    RayD rd;
    for (int k = 0; k < 3; k++) {
        rd.o[k] = C.center[k];
        rd.d[k] = C.dir00[k] + (double)i * C.du[k] + (double)j * C.dv[k];
    }
    rd.time = 0.0;
    Ray ray;
    ray.o = v3((float)rd.o[0], (float)rd.o[1], (float)rd.o[2]);
    ray.d = v3((float)rd.d[0], (float)rd.d[1], (float)rd.d[2]);
    ray.time = 0.0f;
    Hit hit;
    traverse_uploaded(S, ray, 0.001f, __int_as_float(0x7f800000), hit);
    size_t px = (size_t)j * width + i;
    Surface sf;
    sf.prim_id = -1;
    sf.p = sf.normal = v3(0, 0, 0);
    sf.u = sf.v = 0;
    float t = 0.0f;
    if (hit.prim != PRIM_NONE) {
        complete_hit_fp64(S, rd, hit, sf);
        t = sf.t;
    }
    if (prim_id) prim_id[px] = sf.prim_id;
    if (t_out) t_out[px] = t;
    if (normal) { normal[3 * px] = sf.normal.x; normal[3 * px + 1] = sf.normal.y; normal[3 * px + 2] = sf.normal.z; }
    if (point) { point[3 * px] = sf.p.x; point[3 * px + 1] = sf.p.y; point[3 * px + 2] = sf.p.z; }
    if (uv) { uv[2 * px] = sf.u; uv[2 * px + 1] = sf.v; }
}

// Camera.txt:74-89: scale by 1/spp, sqrt gamma, clamp [0, 0.999], int(255.999 * x)
__global__ void resolve_kernel(const unsigned long long* __restrict__ accum, int n_pixels, double inv_scale_spp,
                               float* __restrict__ rgb_linear, unsigned char* __restrict__ rgb8) {
    int px = blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= n_pixels) return;
    for (int c = 0; c < 3; c++) {
        float lin = (float)((double)accum[4ull * px + c] * inv_scale_spp);
        if (rgb_linear) rgb_linear[3ull * px + c] = lin;
        if (rgb8) {
            float g = lin > 0.0f ? sqrtf(lin) : 0.0f;
            g = fminf(fmaxf(g, 0.0f), 0.999f);
            rgb8[3ull * px + c] = (unsigned char)(int)(255.999f * g);
        }
    }
}

// RT_FLAG_MOMENTS resolve.  With n = total_spp, S1 the radiance word and S2 = m0 + m1 * 2^48 its moments (both in the
// 2^-28 units of x), D = n * S2 - S1^2 is computed exactly in 128 bits.  It is >= 0 by Cauchy-Schwarz (dropped samples
// count as x = 0 of the n).  n * S2 can reach 2^128 only when samples saturate at kSampleClamp at 65536 spp: the
// product then saturates at 2^128 - 1 instead of wrapping, and D is a lower bound.
struct U128 {
    unsigned long long lo, hi;
};
__device__ __forceinline__ U128 moments_d(unsigned long long s1, unsigned long long m0, unsigned long long m1, unsigned long long n) {
    const unsigned long long s2_lo = m0 + (m1 << 48);
    const unsigned long long s2_hi = (m1 >> 16) + (s2_lo < m0 ? 1ull : 0ull);
    U128 ns2;
    ns2.lo = n * s2_lo;
    const unsigned long long c = __umul64hi(n, s2_lo);
    ns2.hi = n * s2_hi + c;
    if (__umul64hi(n, s2_hi) != 0 || ns2.hi < c) ns2.lo = ns2.hi = ~0ull;  // saturate
    const unsigned long long q_lo = s1 * s1, q_hi = __umul64hi(s1, s1);
    U128 d;
    if (ns2.hi < q_hi || (ns2.hi == q_hi && ns2.lo < q_lo)) {
        d.lo = d.hi = 0;  // only a total_spp below the true sample count gets here
        return d;
    }
    d.lo = ns2.lo - q_lo;
    d.hi = ns2.hi - q_hi - (ns2.lo < q_lo ? 1ull : 0ull);
    return d;
}
// a 128-bit integer rounded once to the nearest double (ties to even): the top 64 bits with a sticky bit for the rest
__device__ __forceinline__ double u128_to_double(U128 v) {
    if (v.hi == 0) return __ull2double_rn(v.lo);
    const int sh = 64 - __clzll((long long)v.hi);  // 1..64
    const unsigned long long top = sh == 64 ? v.hi : (v.hi << (64 - sh)) | (v.lo >> sh);
    const unsigned long long sticky = (sh == 64 ? v.lo : (v.lo << (64 - sh))) != 0 ? 1ull : 0ull;
    return ldexp(__ull2double_rn(top | sticky), sh);
}
// unbiased per-sample variance s^2 = D / (n (n - 1)) * 2^-56, rounded once to double, divided, rounded once to float
__global__ void variance_kernel(const unsigned long long* __restrict__ accum, const unsigned long long* __restrict__ moments, int n_slots,
                                int n, float* __restrict__ var) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= n_slots) return;
    const double nn1 = (double)n * (double)(n - 1);
    for (int c = 0; c < 3; c++) {
        const U128 d = moments_d(accum[4ull * px + c], moments[6ull * px + 2 * c], moments[6ull * px + 2 * c + 1], (unsigned long long)n);
        var[3ull * px + c] = (float)__dmul_rn(__ddiv_rn(u128_to_double(d), nn1), 0x1p-56);
    }
}
// rt_frame_noise partials, exact integer sums over the slots: out[2c], out[2c + 1] += the low / high 32 bits of S1 of
// channel c; out[6 + 2c], out[7 + 2c] += the low / high 32 bits of q = round(s^2 / n * 2^kNoiseFracBits) of channel c,
// q saturating at 2^64 - 1.  A word adds at most 2^31 values below 2^32: no overflow for any frame rt_render accepts.
constexpr int kNoiseFracBits = 32;
__global__ void noise_kernel(const unsigned long long* __restrict__ accum, const unsigned long long* __restrict__ moments, int n_slots, int n,
                             unsigned long long* __restrict__ out) {
    __shared__ unsigned long long part[12];
    if (threadIdx.x < 12) part[threadIdx.x] = 0;
    __syncthreads();
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long w[12];
    for (int k = 0; k < 12; k++) w[k] = 0;
    if (px < n_slots) {
        const double nn2 = (double)n * (double)n * (double)(n - 1);
        for (int c = 0; c < 3; c++) {
            const unsigned long long s1 = accum[4ull * px + c];
            const U128 d = moments_d(s1, moments[6ull * px + 2 * c], moments[6ull * px + 2 * c + 1], (unsigned long long)n);
            const double q = __dmul_rn(__ddiv_rn(u128_to_double(d), nn2), 0x1p-24);  // s^2 / n in 2^-kNoiseFracBits units
            const unsigned long long qi = q >= 0x1p64 ? ~0ull : __double2ull_rn(q);
            w[2 * c] = s1 & 0xffffffffull;
            w[2 * c + 1] = s1 >> 32;
            w[6 + 2 * c] = qi & 0xffffffffull;
            w[7 + 2 * c] = qi >> 32;
        }
    }
    for (int k = 0; k < 12; k++) {
        unsigned long long v = w[k];
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31u) == 0 && v) atomicAdd(&part[k], v);
    }
    __syncthreads();
    if (threadIdx.x < 12 && part[threadIdx.x]) atomicAdd(out + threadIdx.x, part[threadIdx.x]);
}

__global__ void probe_texture_kernel(const __grid_constant__ DevScene S, int tex, int n, const float* __restrict__ uvp,
                                     float* __restrict__ rgb) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    V3 c = tex_value(S, tex, uvp[5 * i], uvp[5 * i + 1], v3(uvp + 5 * i + 2));
    rgb[3 * i] = c.x; rgb[3 * i + 1] = c.y; rgb[3 * i + 2] = c.z;
}

__global__ void probe_scatter_kernel(const __grid_constant__ DevScene S, int mat, int n, const float* __restrict__ in,
                                     const float* __restrict__ uni, float* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* r = in + 16 * (size_t)i;
    Ray ray;
    ray.o = v3(r); ray.d = v3(r + 3); ray.time = r[6];
    Surface sf;
    sf.p = v3(r + 7); sf.normal = v3(r + 10); sf.front = r[13] != 0.0f; sf.u = r[14]; sf.v = r[15];
    sf.material = mat; sf.prim_id = -1;
    const DevMaterial& m = S.mats[mat];
    V3 em = mat_emitted(S, m, sf);
    float4 u4 = make_float4(uni[4 * i], uni[4 * i + 1], uni[4 * i + 2], uni[4 * i + 3]);
    V3 att = v3(0, 0, 0);
    Ray next;
    next.o = next.d = v3(0, 0, 0);
    next.time = 0;
    bool ok = mat_scatter(S, m, ray, sf, u4, att, next);
    float* o = out + 16 * (size_t)i;
    o[0] = ok ? 1.0f : 0.0f;
    o[1] = att.x; o[2] = att.y; o[3] = att.z;
    o[4] = next.o.x; o[5] = next.o.y; o[6] = next.o.z;
    o[7] = next.d.x; o[8] = next.d.y; o[9] = next.d.z;
    o[10] = em.x; o[11] = em.y; o[12] = em.z;
    o[13] = next.time; o[14] = o[15] = 0.0f;
}

__global__ void probe_hit_kernel(const __grid_constant__ DevScene S, int n, const float* __restrict__ rays, int* __restrict__ prim_id,
                                 float* __restrict__ t_out, float* __restrict__ normal, float* __restrict__ uv) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* r = rays + 9 * (size_t)i;
    Ray ray;
    ray.o = v3(r); ray.d = v3(r + 3); ray.time = r[6];
    Hit hit;
    traverse_uploaded(S, ray, r[7], r[8], hit);
    Surface sf;
    sf.prim_id = -1;
    sf.normal = v3(0, 0, 0);
    sf.u = sf.v = 0;
    sf.t = 0.0f;
    if (hit.prim != PRIM_NONE) complete_hit(S, ray, hit, sf, true);  // exactly what the render kernels compute (FP32, FP64 sphere refinement)
    if (prim_id) prim_id[i] = sf.prim_id;
    if (t_out) t_out[i] = sf.t;
    if (normal) { normal[3 * i] = sf.normal.x; normal[3 * i + 1] = sf.normal.y; normal[3 * i + 2] = sf.normal.z; }
    if (uv) { uv[2 * i] = sf.u; uv[2 * i + 1] = sf.v; }
}

// 8 independent FMA chains per thread: measures the FP32 issue roof (2 flops per FMA)
__global__ void fma_peak_kernel(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
        x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
    float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678f) out[0] = s;
}

// L1 load bandwidth: every warp streams 128-bit loads over a 32 KB window of its block (L1-resident after the
// first sweep), four independent accumulators per thread.  The denominator of the node/primitive-bytes figure:
// the BASELINE scenes live in L1/L2, so their bytes per second are a cache-bandwidth number, not an HBM one.
__global__ void l1_peak_kernel(const uint4* __restrict__ buf, int iters, uint4* __restrict__ out) {
    const uint4* base = buf + (size_t)blockIdx.x * 2048;  // 2048 x 16 B = 32 KB per block
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0, a2 = a0, a3 = a0;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
            // the window position moves with the iteration: loop-invariant addresses would be hoisted
            const unsigned at = threadIdx.x + (unsigned)(8 * i + 4 * k) * 256u;
            const uint4 v0 = __ldca(base + (at & 2047u));
            const uint4 v1 = __ldca(base + ((at + 256u) & 2047u));
            const uint4 v2 = __ldca(base + ((at + 512u) & 2047u));
            const uint4 v3 = __ldca(base + ((at + 768u) & 2047u));
            a0.x ^= v0.x; a0.y ^= v0.y; a0.z ^= v0.z; a0.w ^= v0.w;
            a1.x ^= v1.x; a1.y ^= v1.y; a1.z ^= v1.z; a1.w ^= v1.w;
            a2.x ^= v2.x; a2.y ^= v2.y; a2.z ^= v2.z; a2.w ^= v2.w;
            a3.x ^= v3.x; a3.y ^= v3.y; a3.z ^= v3.z; a3.w ^= v3.w;
        }
        asm volatile("" ::: "memory");
    }
    const uint4 r = make_uint4(a0.x ^ a1.x ^ a2.x ^ a3.x, a0.y ^ a1.y ^ a2.y ^ a3.y, a0.z ^ a1.z ^ a2.z ^ a3.z, a0.w ^ a1.w ^ a2.w ^ a3.w);
    if (r.x == 0x12345678u && r.y == 0x9abcdef0u) out[0] = r;
}

// ---------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------
// Layout of an accumulation buffer.  Full: one 32-byte slot per pixel, row-major.  Compact
// (RT_FLAG_COMPACT_TILES): only the tiles of one shard (tile t of the frame belongs to shard t mod count
// and is its local tile t / count), each tile a tile_size x tile_size block of slots -- 1 / count of the
// frame, which is what a GPU of a tile-sharded frame needs and what travels in the gather.
struct AccumLayout {
    int width = 0, height = 0;
    bool compact = false;
    int rank = 0, count = 1, tile = 16;
    bool operator==(const AccumLayout& o) const {
        return width == o.width && height == o.height && compact == o.compact && (!compact || (rank == o.rank && count == o.count && tile == o.tile));
    }
    size_t local_tiles() const {
        const size_t tiles = (size_t)((width + tile - 1) / tile) * ((height + tile - 1) / tile);
        return tiles > (size_t)rank ? (tiles - rank + count - 1) / count : 0;
    }
    size_t slots() const { return compact ? local_tiles() * tile * tile : (size_t)width * height; }
    // pixels of the frame the slots hold (a compact buffer's partial edge tiles have slots outside the frame)
    size_t pixels() const {
        if (!compact) return (size_t)width * height;
        const int tiles_x = (width + tile - 1) / tile, n_tiles = tiles_x * ((height + tile - 1) / tile);
        size_t px = 0;
        for (int t = rank; t < n_tiles; t += count)
            px += (size_t)std::min(tile, width - (t % tiles_x) * tile) * std::min(tile, height - (t / tiles_x) * tile);
        return px;
    }
};

struct DevCtx {
    int device = 0;
    std::string error;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // the whole device scene lives in ONE arena, staged in pinned host memory and moved with
    // one copy per rt_upload_scene; both grow on demand and are reused across uploads
    unsigned char* arena = nullptr;
    size_t arena_cap = 0;
    unsigned char* staging = nullptr;
    size_t staging_cap = 0;
    // persistent output buffers of rt_download
    float* out_lin = nullptr;
    unsigned char* out_rgb8 = nullptr;
    size_t out_pixels = 0;
    DevScene scene{};
    bool has_scene = false;
    bool scene_lite = false;  // no triangles, no point lights, no defocus: the LITE kernel instance applies
    bool geom_lite = false;   // no triangles, no point lights: LITE up to the camera (rt_render_views checks its views)
    rt_camera camera{};
    // accumulation
    unsigned long long* accum = nullptr;
    size_t accum_bytes = 0, accum_cap = 0;
    bool accum_external = false;
    AccumLayout acc;                        // layout of `accum`
    // RT_FLAG_MOMENTS: 6 words per slot of `acc` (add_square), allocated by the first moments render; valid when they
    // describe the same samples as the sums (set by a non-accumulating moments pass or rt_moments_upload, cleared by
    // an accumulating pass without the flag, a pass that replaces the frame without it, a layout change, rt_bind_accum
    // and rt_accum_upload)
    unsigned long long* moments = nullptr;
    size_t moments_cap = 0;
    bool moments_valid = false;
    bool sums_uploaded = false;              // the frame is an rt_accum_upload, not rendered onto since (rt_moments_upload)
    unsigned long long* noise_sums = nullptr;  // rt_frame_noise: the 12 partial words of noise_kernel
    // rt_render_views: the views frame (views_n x views_h x views_w slots of 32 B, view-major; no other call touches it),
    // the view table on the device, and what an accumulating views pass must match: the frame's shape and a
    // fingerprint of the cameras and seeds (views_n == 0: no views render yet)
    unsigned long long* views_accum = nullptr;
    size_t views_cap = 0;
    ViewRecord* view_table = nullptr;
    size_t view_table_cap = 0;
    int views_n = 0, views_w = 0, views_h = 0;
    uint64_t views_key = 0;
    unsigned char* frame_scratch = nullptr;  // full-frame copies of compact data (checkpoints, single-shard downloads)
    size_t frame_scratch_cap = 0;
    unsigned long long* counters = nullptr;  // [0] work counter, [1..3] unused
    Stats* dstats = nullptr;
    rt_stats stats{};
    int cam_w = 0, cam_h = 0;  // frame the device camera block was computed for
    CameraD camera_d{};        // the same camera in double (deterministic pixel-centre rays of the AOV)
    int sm_count = 0;
    // acceleration structure the render kernels traverse: 2 = binary tree, 8 / 4 = wide quantised tree
    // (host-built scenes only; a device-built scene keeps the binary tree).  rt_set_bvh_width / RT_B200_BVH_WIDTH
    // asynchronous frame hand-out (rt_download_begin / rt_untile_begin / rt_frame_end): the device-to-host copy runs on
    // its own stream into pinned double buffers while the next pass renders
    struct OutFrame {
        cudaEvent_t done = nullptr;
        unsigned char* pinned = nullptr;
        size_t cap = 0, off_lin = 0, off_rgb8 = 0;
        bool has_lin = false, has_rgb8 = false, active = false;
    };
    OutFrame frames[2];
    int frame_head = 0, frames_out = 0;  // next slot to fill, outstanding begins
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_ready = nullptr;       // the device-side frame (resolved / untiled) is complete
    int n_materials = 0, n_textures = 0;  // sizes of the uploaded tables (the probes check their indices)
    uint64_t staged_key = 0;   // fingerprint of the scene whose arena image is in `staging` (0: none)
    size_t staged_bytes = 0;
    int bvh_width = RT_B200_DEFAULT_BVH_WIDTH;
    int scene_feat = FEAT_ALL;  // FEAT_* bits the uploaded scene needs
    int wide_depth = 0;  // levels of the uploaded wide tree = stack entries a ray can need
    // RT_FLAG_OVERLAP: asynchronous accumulate passes alternate between two streams of the context, each with its own work
    // counter (counters + 4 and + 8), so that the drain of one pass runs while the next takes over the freed SM slots
    cudaStream_t lane_stream[2] = {nullptr, nullptr};
    cudaEvent_t lane_end[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ov_begin = nullptr;
    bool lane_busy[2] = {false, false};
    int lane_next = 0, ov_passes = 0;
    bool pending_async = false;           // an RT_FLAG_ASYNC render has not been waited for yet (dev_wait)
    bool pending_stats = false;
    cudaStream_t pending_stream = nullptr;  // the stream it was enqueued on
    // scene-upload path: 0 auto (device from kDeviceBuildAuto primitives up), 1 host SAH, 2 device (LBVH + SAH top levels), 3 device, pure LBVH
    int bvh_builder = 0;
    size_t world_type_count[4] = {0, 0, 0, 0};  // primitives of each device type in the world list (validate_scene)
    int n_prims = 0;  // primitives of the world list with every mesh ref expanded to its triangles (validate_scene)
    rtlbvh::CopyRing copy_ring;        // pinned staging of the device path's raw-input copy
    unsigned char* scratch = nullptr;  // work space of the device build and of rt_refit_scene, reused across calls
    size_t scratch_cap = 0;
    // the scene-side state of the scene whose arena image is in `staging`: a cache hit of rt_upload_scene restores it
    // together with the arena (an rt_refit_scene in between changes both)
    struct SceneState {
        DevScene scene;
        rt_camera camera;
        int scene_feat;
        bool scene_lite, geom_lite;
    } staged_state{};
    // what rt_refit_scene compares a description with: the structure of the uploaded scene
    struct Shape {
        int32_t counts[13];
        std::vector<int32_t> mesh_tris, image_wh;
        std::vector<uint32_t> boundary_packed;  // the boundaries' records (type << 28 | index)
        std::vector<int8_t> media_class;        // 1 one sphere, 2 a six-quad box, 0 general
        // the next-event emitters in list order: canonical ids of a host-built scene, source quads of a device-built one
        std::vector<int32_t> nee_ids;
        std::vector<unsigned char*> image_dev;  // the images' texels in the arena
        int n_prims;                             // world primitives with the meshes expanded, and of each device type
        size_t world_type_count[4];
        bool device_built;                       // the tree and the world records were built on the device
    } shape;
    rtlbvh::RefitTree refit_tree;  // the uploaded tree in the order the refit visits it (derived on its first refit)
};

// From this many primitives on, RT_B200_BVH=auto builds on the device: the host SAH build costs
// ~0.4 ms per thousand triangles (30 ms at this size), the device path ~2 ms, and with the
// per-cluster SAH rebuild and the SAH top levels the device-built tree traces within -1...-12 % of
// the host's (DESIGN.md section 10).  Every BASELINE scene is smaller and keeps the host tree.
constexpr int kDeviceBuildAuto = 1 << 16;
// the wide kernels keep their traversal stack in shared memory: 8 bytes x threads x levels per block
constexpr int kWideMaxDepth = 24;
constexpr int kDeviceBuildMin = 8;

static int fail(DevCtx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->error = buf;
    return code;
}

#define CU(ctx, call)                                                                                       \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) return fail(ctx, RT_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));      \
    } while (0)

static void free_scene(DevCtx* ctx) { ctx->has_scene = false; }

static void release_buffers(DevCtx* ctx) {
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->scratch) cudaFree(ctx->scratch);
    ctx->copy_ring.release();
    ctx->refit_tree.release();
    ctx->scratch = nullptr;
    ctx->scratch_cap = 0;
    if (ctx->staging) cudaFreeHost(ctx->staging);
    if (ctx->out_lin) cudaFree(ctx->out_lin);
    if (ctx->out_rgb8) cudaFree(ctx->out_rgb8);
    if (ctx->frame_scratch) cudaFree(ctx->frame_scratch);
    ctx->frame_scratch = nullptr;
    ctx->frame_scratch_cap = 0;
    ctx->arena = ctx->staging = ctx->out_rgb8 = nullptr;
    ctx->out_lin = nullptr;
    ctx->arena_cap = ctx->staging_cap = ctx->out_pixels = 0;
}

// layout of the scene arena: every block 256-byte aligned
struct ArenaPlan {
    size_t size = 0;
    size_t add(size_t bytes) {
        size_t off = (size + 255) & ~(size_t)255;
        size = off + std::max<size_t>(bytes, 16);
        return off;
    }
};

static int dev_create(DevCtx** out, const int* device_ids, int n_devices) {
    if (!out) return RT_ERR_INVALID;
    *out = nullptr;
    DevCtx* ctx = new (std::nothrow) DevCtx();
    if (!ctx) return RT_ERR_NOMEM;
    *out = ctx;  // returned even on failure so that rt_last_error works; caller destroys it
    if (n_devices != 1 || !device_ids) return fail(ctx, RT_ERR_INVALID, "rt_create: exactly one device per context (got %d)", n_devices);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(ctx, RT_ERR_CUDA, "rt_create: no CUDA device (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    ctx->device = device_ids[0];
    if (ctx->device < 0 || ctx->device >= count) return fail(ctx, RT_ERR_INVALID, "rt_create: device %d out of range", ctx->device);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CU(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    if (prop.major < 10) return fail(ctx, RT_ERR_CUDA, "rt_create: device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    CU(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(ctx, cudaEventCreate(&ctx->ev0));
    CU(ctx, cudaEventCreate(&ctx->ev1));
    CU(ctx, cudaMalloc(&ctx->counters, 12 * sizeof(unsigned long long)));  // {work counter, -, -, -} x (plain, overlap lane 0, lane 1)
    CU(ctx, cudaMalloc(&ctx->dstats, sizeof(Stats) + kTravHistBins * sizeof(unsigned long long)));
    // local-memory traversal stacks live in L1: prefer L1 over shared memory (the wide instances
    // get their carve-out per launch, from the depth of the uploaded tree)
    for (const V2Instance& e : kV2Instances)
        if (e.width == 2) cudaFuncSetAttribute((const void*)e.kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    if (const char* bv = getenv("RT_B200_BVH"))
        ctx->bvh_builder = strcmp(bv, "host") == 0 ? 1 : (strcmp(bv, "device") == 0 ? 2 : (strcmp(bv, "lbvh") == 0 ? 3 : 0));
    if (const char* wv = getenv("RT_B200_BVH_WIDTH")) {
        const int w = atoi(wv);
        if (w != 2 && w != 4 && w != 8) return fail(ctx, RT_ERR_INVALID, "RT_B200_BVH_WIDTH=%s: 2, 4 or 8", wv);
        ctx->bvh_width = w;
    }
    if (const char* kv = getenv("RT_B200_KERNEL"))
        if (strcmp(kv, "v2") != 0)
            return fail(ctx, RT_ERR_UNSUPPORTED, "RT_B200_KERNEL=%s: render_kernel_v2 is the only render kernel; the alternatives were removed (DESIGN.md section 3)", kv);
    cudaFuncAttributes fa;
    CU(ctx, cudaFuncGetAttributes(&fa, render_kernel_v2<false, false>));
    ctx->stats.regs_per_thread = fa.numRegs;
    ctx->stats.local_bytes_per_thread = (uint32_t)fa.localSizeBytes;
    ctx->stats.threads_per_block = RT_V2_THREADS;
    return RT_OK;
}

static void dev_destroy(DevCtx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    free_scene(ctx);
    release_buffers(ctx);
    if (ctx->accum && !ctx->accum_external) cudaFree(ctx->accum);
    if (ctx->moments) cudaFree(ctx->moments);
    if (ctx->noise_sums) cudaFree(ctx->noise_sums);
    if (ctx->views_accum) cudaFree(ctx->views_accum);
    if (ctx->view_table) cudaFree(ctx->view_table);
    if (ctx->counters) cudaFree(ctx->counters);
    if (ctx->dstats) cudaFree(ctx->dstats);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (int k = 0; k < 2; k++) {
        if (ctx->lane_stream[k]) { cudaStreamSynchronize(ctx->lane_stream[k]); cudaStreamDestroy(ctx->lane_stream[k]); }
        if (ctx->lane_end[k]) cudaEventDestroy(ctx->lane_end[k]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ov_begin) cudaEventDestroy(ctx->ov_begin);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->ev_ready) cudaEventDestroy(ctx->ev_ready);
    for (auto& f : ctx->frames) {
        if (f.done) cudaEventDestroy(f.done);
        if (f.pinned) cudaFreeHost(f.pinned);
    }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}


// ---------------------------------------------------------------------------------
// scene upload
// ---------------------------------------------------------------------------------
namespace {

using rtprep::BakedPrim;
using rtprep::D3;
using rtprep::d3;
using rtprep::dcross;
using rtprep::ddot;
using rtprep::dunit;
using rtprep::xf_dir;
using rtprep::xf_point;
using rtprep::operator+;
using rtprep::operator-;
using rtprep::operator*;
static_assert((uint32_t)rtprep::PREP_SPHERE == (uint32_t)PT_SPHERE && (uint32_t)rtprep::PREP_MSPHERE == (uint32_t)PT_MSPHERE &&
              (uint32_t)rtprep::PREP_QUAD == (uint32_t)PT_QUAD && (uint32_t)rtprep::PREP_TRI == (uint32_t)PT_TRI, "primitive type codes");

bool texture_needs_uv(const rt_scene_desc* sc, int tex, int depth = 0) {
    if (tex < 0 || tex >= sc->n_textures || depth > 16) return false;
    const rt_texture& t = sc->textures[tex];
    if (t.type == RT_TEX_IMAGE || t.type == RT_TEX_CHECKER_TRIANGLE) return true;
    if (t.type == RT_TEX_CHECKER) return texture_needs_uv(sc, t.even, depth + 1) || texture_needs_uv(sc, t.odd, depth + 1);
    return false;
}

// the first of n triangles with a corner index >= bound, or -1; big index buffers are split over the host cores
int first_bad_triangle(const uint32_t* idx, int n, uint32_t bound) {
    const int workers = n < (1 << 18) ? 1 : (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<int> bad((size_t)workers, -1);
    auto run = [&](int w) {
        const int a = (int)((long long)n * w / workers), b = (int)((long long)n * (w + 1) / workers);
        for (int t = a; t < b; t++) {
            const uint32_t* c = idx + 3 * (size_t)t;
            if ((c[0] >= bound) | (c[1] >= bound) | (c[2] >= bound)) { bad[(size_t)w] = t; return; }
        }
    };
    std::vector<std::thread> pool;
    for (int w = 1; w < workers; w++) pool.emplace_back(run, w);
    run(0);
    for (auto& t : pool) t.join();
    for (int b : bad)
        if (b >= 0) return b;
    return -1;
}

}  // namespace

// shallow: what must hold before the arrays may be read at all (the fingerprint of an unchanged scene is taken next);
// the full pass checks every index
static int validate_scene(DevCtx* ctx, const rt_scene_desc* sc, bool shallow) {
    if (!sc) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: null scene");
    if (sc->struct_size != sizeof(rt_scene_desc) || sc->abi_version != RT_B200_ABI_VERSION)
        return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: ABI mismatch (struct_size %u vs %zu, abi %u vs %d)", sc->struct_size,
                    sizeof(rt_scene_desc), sc->abi_version, RT_B200_ABI_VERSION);
    auto neg = [](int n) { return n < 0; };
    if (neg(sc->n_world) || neg(sc->n_boundary_refs) || neg(sc->n_spheres) || neg(sc->n_quads) || neg(sc->n_triangles) ||
        neg(sc->n_media) || neg(sc->n_xforms) || neg(sc->n_materials) || neg(sc->n_textures) || neg(sc->n_images) ||
        neg(sc->n_perlins) || neg(sc->n_lights) || neg(sc->n_meshes))
        return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: negative count");
    if ((long long)sc->n_world + sc->n_boundary_refs >= (1 << 25)) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_upload_scene: more than 2^25 primitives");
    // every array with a non-zero count must be there: nothing below dereferences a null pointer
    if ((sc->n_world && !sc->world) || (sc->n_boundary_refs && !sc->boundary_refs) || (sc->n_spheres && !sc->spheres) || (sc->n_quads && !sc->quads) ||
        (sc->n_triangles && !sc->triangles) || (sc->n_media && !sc->media) || (sc->n_xforms && !sc->xforms) || (sc->n_materials && !sc->materials) ||
        (sc->n_textures && !sc->textures) || (sc->n_images && !sc->images) || (sc->n_perlins && !sc->perlins) || (sc->n_lights && !sc->lights) ||
        (sc->n_meshes && !sc->meshes))
        return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: an array with a non-zero count is null");
    for (int i = 0; i < sc->n_meshes; i++) {
        const rt_mesh& m = sc->meshes[i];
        if (neg(m.n_vertices) || neg(m.n_triangles) || neg(m.n_uvs)) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: negative count", i);
        if ((m.n_vertices && !m.positions) || (m.n_triangles && !m.indices) || (m.n_uvs && !m.uvs) || (m.uv_indices && !m.uvs))
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: an array with a non-zero count is null (or uv_indices without uvs)", i);
        if (m.uvs && !m.uv_indices && m.n_uvs != m.n_vertices)
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: without uv_indices n_uvs (%d) must equal n_vertices (%d)", i, m.n_uvs, m.n_vertices);
        if (m.material < 0 || m.material >= sc->n_materials) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: material out of range", i);
        if (m.xform < -1 || m.xform >= sc->n_xforms) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: xform out of range", i);
    }
    // the primitive count: a mesh ref stands for its triangles (a bad ref counts one here and is refused by the full pass)
    long long n_prims = sc->n_world;
    if (sc->n_meshes > 0) {
        n_prims = 0;
        for (int i = 0; i < sc->n_world; i++) {
            const rt_prim_ref r = sc->world[i];
            n_prims += (r.type == RT_PRIM_MESH && r.index >= 0 && r.index < sc->n_meshes) ? sc->meshes[r.index].n_triangles : 1;
        }
    }
    if (n_prims + sc->n_boundary_refs >= (1 << 25))
        return fail(ctx, RT_ERR_UNSUPPORTED, "rt_upload_scene: more than 2^25 primitives (%lld with the meshes expanded)", n_prims + sc->n_boundary_refs);
    ctx->n_prims = (int)n_prims;
    // the free-flight uniforms of medium m come from Philox stream RS_MEDIUM + m / 4, which shares its counter word with
    // the bounce number shifted by 8: more media than this would run into the bounce bits
    if (sc->n_media > 4 * (256 - (int)RS_MEDIUM)) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_upload_scene: at most %d media", 4 * (256 - (int)RS_MEDIUM));
    if (shallow) return RT_OK;
    auto check_ref = [&](const rt_prim_ref& r, bool boundary) -> const char* {
        if (r.type == RT_PRIM_MESH && !boundary) return r.index < 0 || r.index >= sc->n_meshes ? "mesh index out of range" : nullptr;
        int n = r.type == RT_PRIM_SPHERE ? sc->n_spheres : r.type == RT_PRIM_QUAD ? sc->n_quads : r.type == RT_PRIM_TRIANGLE ? sc->n_triangles : -1;
        if (n < 0) return "unknown primitive type";
        if (r.index < 0 || r.index >= n) return "primitive index out of range";
        int mat = r.type == RT_PRIM_SPHERE ? sc->spheres[r.index].material : r.type == RT_PRIM_QUAD ? sc->quads[r.index].material : sc->triangles[r.index].material;
        int xf = r.type == RT_PRIM_SPHERE ? sc->spheres[r.index].xform : r.type == RT_PRIM_QUAD ? sc->quads[r.index].xform : sc->triangles[r.index].xform;
        if (!boundary && (mat < 0 || mat >= sc->n_materials)) return "material index out of range";
        if (xf < -1 || xf >= sc->n_xforms) return "xform index out of range";
        return nullptr;
    };
    // the world list is the one O(n) part of validation: big scenes split it over the host cores,
    // and count the primitives of each DEVICE type on the way (the device upload path sizes its
    // arena blocks from these counts)
    {
        const int n = sc->n_world;
        const int workers = n < (1 << 16) ? 1 : (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        struct Part { int bad = -1; const char* msg = nullptr; size_t count[4] = {0, 0, 0, 0}; };
        std::vector<Part> parts((size_t)workers);
        auto run = [&](int w) {
            Part& p = parts[(size_t)w];
            const int a = (int)((long long)n * w / workers), b = (int)((long long)n * (w + 1) / workers);
            for (int i = a; i < b; i++) {
                const rt_prim_ref r = sc->world[i];
                if (const char* m = check_ref(r, false)) { p.bad = i; p.msg = m; return; }
                if (r.type == RT_PRIM_MESH) {
                    p.count[PT_TRI] += (size_t)sc->meshes[r.index].n_triangles;
                    continue;
                }
                uint32_t t = r.type == RT_PRIM_QUAD ? PT_QUAD : (r.type == RT_PRIM_TRIANGLE ? PT_TRI : PT_SPHERE);
                if (r.type == RT_PRIM_SPHERE) {
                    const double* v = sc->spheres[r.index].center_vec;
                    if (v[0] != 0 || v[1] != 0 || v[2] != 0) t = PT_MSPHERE;
                }
                p.count[t]++;
            }
        };
        if (workers == 1) {
            run(0);
        } else {
            std::vector<std::thread> pool;
            for (int w = 1; w < workers; w++) pool.emplace_back(run, w);
            run(0);
            for (auto& t : pool) t.join();
        }
        for (int k = 0; k < 4; k++) ctx->world_type_count[k] = 0;
        for (const Part& p : parts) {
            if (p.bad >= 0) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: world[%d]: %s", p.bad, p.msg);
            for (int k = 0; k < 4; k++) ctx->world_type_count[k] += p.count[k];
        }
    }
    for (int i = 0; i < sc->n_boundary_refs; i++) {
        if (sc->boundary_refs[i].type == RT_PRIM_MESH) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_upload_scene: boundary_refs[%d]: a mesh cannot bound a medium", i);
        if (const char* m = check_ref(sc->boundary_refs[i], true)) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: boundary_refs[%d]: %s", i, m);
    }
    // every mesh index, before anything gathers through it (host or device path)
    for (int i = 0; i < sc->n_meshes; i++) {
        const rt_mesh& m = sc->meshes[i];
        int tri = -1;
        if ((tri = first_bad_triangle(m.indices, m.n_triangles, (uint32_t)m.n_vertices)) >= 0)
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: triangle %d: position index out of range (n_vertices %d)", i, tri, m.n_vertices);
        if (m.uv_indices && (tri = first_bad_triangle(m.uv_indices, m.n_triangles, (uint32_t)m.n_uvs)) >= 0)
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: meshes[%d]: triangle %d: uv index out of range (n_uvs %d)", i, tri, m.n_uvs);
    }
    for (int i = 0; i < sc->n_media; i++) {
        const rt_medium& m = sc->media[i];
        if (m.boundary_first < 0 || m.boundary_count < 0 || m.boundary_first + m.boundary_count > sc->n_boundary_refs)
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: media[%d]: boundary range out of bounds", i);
        if (m.material < 0 || m.material >= sc->n_materials) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: media[%d]: material out of range", i);
        if (!(m.density > 0) || m.multiplicity < 1) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: media[%d]: density/multiplicity must be positive", i);
        if (m.xform < -1 || m.xform >= sc->n_xforms) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: media[%d]: xform out of range", i);
    }
    for (int i = 0; i < sc->n_materials; i++) {
        const rt_material& m = sc->materials[i];
        if (m.type < RT_MAT_LAMBERTIAN || m.type > RT_MAT_SPECULAR) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: materials[%d]: unknown type %d", i, m.type);
        bool textured = m.type == RT_MAT_LAMBERTIAN || m.type == RT_MAT_DIFFUSE_LIGHT || m.type == RT_MAT_EMISSIVE_LIGHT || m.type == RT_MAT_ISOTROPIC;
        if (textured && (m.texture < 0 || m.texture >= sc->n_textures)) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: materials[%d]: texture out of range", i);
    }
    for (int i = 0; i < sc->n_textures; i++) {
        const rt_texture& t = sc->textures[i];
        if (t.type < RT_TEX_SOLID || t.type > RT_TEX_NOISE) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: textures[%d]: unknown type %d", i, t.type);
        if ((t.type == RT_TEX_CHECKER || t.type == RT_TEX_CHECKER_TRIANGLE) && (t.even < 0 || t.even >= sc->n_textures || t.odd < 0 || t.odd >= sc->n_textures))
            return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: textures[%d]: child out of range", i);
        if (t.type == RT_TEX_IMAGE && t.image >= sc->n_images) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: textures[%d]: image out of range", i);
        if (t.type == RT_TEX_NOISE && (t.perlin < 0 || t.perlin >= sc->n_perlins)) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: textures[%d]: perlin out of range", i);
    }
    for (int i = 0; i < sc->n_images; i++)
        if (sc->images[i].width <= 0 || sc->images[i].height <= 0 || !sc->images[i].rgb) return fail(ctx, RT_ERR_INVALID, "rt_upload_scene: images[%d]: empty", i);
    return RT_OK;
}

// A 64-bit fingerprint of everything rt_upload_scene reads (the description, the arrays behind it, the texels) and
// of the builder settings: an upload of the SAME scene (camera::render in a loop, progressive passes that re-upload)
// skips validation, transform baking, the BVH build and the record derivation and only repeats the copy of the staged
// arena to the device.  Word-wise multiply-xorshift (~5 GB/s); a collision would need 2^-64 luck.
static uint64_t hash_bytes(uint64_t h, const void* data, size_t bytes) {
    const unsigned char* p = (const unsigned char*)data;
    const uint64_t k = 0x9E3779B97F4A7C15ull;
    size_t i = 0;
    for (; i + 8 <= bytes; i += 8) {
        uint64_t w;
        std::memcpy(&w, p + i, 8);
        h = (h ^ w) * k;
        h ^= h >> 29;
    }
    uint64_t tail = 0;
    if (i < bytes) std::memcpy(&tail, p + i, bytes - i);
    h = (h ^ tail ^ ((uint64_t)bytes << 56)) * k;
    return h ^ (h >> 32);
}
static uint64_t scene_key(const DevCtx* ctx, const rt_scene_desc* sc) {
    uint64_t h = 0x1234567887654321ull;
    const int32_t counts[16] = {sc->n_world, sc->n_boundary_refs, sc->n_spheres, sc->n_quads, sc->n_triangles, sc->n_media, sc->n_xforms, sc->n_materials,
                                sc->n_textures, sc->n_images, sc->n_perlins, sc->n_lights, ctx->bvh_builder, ctx->bvh_width, RT_B200_ABI_VERSION, sc->n_meshes};
    h = hash_bytes(h, counts, sizeof counts);
    h = hash_bytes(h, &sc->camera, sizeof sc->camera);
    h = hash_bytes(h, sc->world, (size_t)sc->n_world * sizeof(rt_prim_ref));
    h = hash_bytes(h, sc->boundary_refs, (size_t)sc->n_boundary_refs * sizeof(rt_prim_ref));
    h = hash_bytes(h, sc->spheres, (size_t)sc->n_spheres * sizeof(rt_sphere));
    h = hash_bytes(h, sc->quads, (size_t)sc->n_quads * sizeof(rt_quad));
    h = hash_bytes(h, sc->triangles, (size_t)sc->n_triangles * sizeof(rt_triangle));
    h = hash_bytes(h, sc->media, (size_t)sc->n_media * sizeof(rt_medium));
    h = hash_bytes(h, sc->xforms, (size_t)sc->n_xforms * sizeof(rt_xform));
    h = hash_bytes(h, sc->materials, (size_t)sc->n_materials * sizeof(rt_material));
    h = hash_bytes(h, sc->textures, (size_t)sc->n_textures * sizeof(rt_texture));
    h = hash_bytes(h, sc->perlins, (size_t)sc->n_perlins * sizeof(rt_perlin));
    h = hash_bytes(h, sc->lights, (size_t)sc->n_lights * sizeof(rt_point_light));
    for (int i = 0; i < sc->n_meshes; i++) {
        const rt_mesh& m = sc->meshes[i];
        const int32_t f[6] = {m.n_vertices, m.n_triangles, m.n_uvs, m.material, m.xform, (m.uvs ? 1 : 0) | (m.uv_indices ? 2 : 0)};
        h = hash_bytes(h, f, sizeof f);
        h = hash_bytes(h, m.positions, (size_t)m.n_vertices * 3 * sizeof(float));
        h = hash_bytes(h, m.indices, (size_t)m.n_triangles * 3 * sizeof(uint32_t));
        if (m.uvs) h = hash_bytes(h, m.uvs, (size_t)m.n_uvs * 2 * sizeof(float));
        if (m.uv_indices) h = hash_bytes(h, m.uv_indices, (size_t)m.n_triangles * 3 * sizeof(uint32_t));
    }
    for (int i = 0; i < sc->n_images; i++) {
        const int32_t wh[2] = {sc->images[i].width, sc->images[i].height};
        h = hash_bytes(h, wh, sizeof wh);
        if (sc->images[i].rgb && wh[0] > 0 && wh[1] > 0) h = hash_bytes(h, sc->images[i].rgb, (size_t)wh[0] * wh[1] * 3);
    }
    return h ? h : 1;
}

// Camera.txt:136-175 in double for a width x height frame: the FP32 camera block the render kernels read (fields named
// as in DevScene and ViewRecord) and the same vectors in double for the AOV.  A pure function of (camera, width,
// height): rt_render and every view of rt_render_views get the same floats from the same operations in the same order,
// which is what makes a view bit-identical to a single render with that camera.
struct CameraBlock {
    float center[3], dir00[3], du[3], dv[3], disk_u[3], disk_v[3];
    int defocus;
    CameraD d;
};
static CameraBlock camera_block(const rt_camera& c, int width, int height) {
    const double pi = 3.1415926535897932385;
    D3 lookfrom = d3(c.lookfrom), lookat = d3(c.lookat), vup = d3(c.vup);
    double theta = c.vfov * pi / 180.0;
    double h = std::tan(theta / 2);
    double viewport_height = 2 * h * c.focus_dist;
    double viewport_width = viewport_height * (double(width) / height);
    D3 w = dunit(lookfrom - lookat);
    D3 u = dunit(dcross(vup, w));
    D3 v = dcross(w, u);
    D3 viewport_u = viewport_width * u;
    D3 viewport_v = viewport_height * (-1.0 * v);
    D3 du = (1.0 / width) * viewport_u;
    D3 dv = (1.0 / height) * viewport_v;
    // pixel00_loc - center
    D3 dir00 = (-c.focus_dist) * w - 0.5 * viewport_u - 0.5 * viewport_v + 0.5 * (du + dv);
    double defocus_radius = c.focus_dist * std::tan((c.defocus_angle / 2) * pi / 180.0);
    D3 disk_u = defocus_radius * u, disk_v = defocus_radius * v;
    CameraBlock B;
    auto put = [](float* dst, D3 s) { dst[0] = (float)s.x; dst[1] = (float)s.y; dst[2] = (float)s.z; };
    put(B.center, lookfrom);
    put(B.dir00, dir00);
    put(B.du, du);
    put(B.dv, dv);
    put(B.disk_u, disk_u);
    put(B.disk_v, disk_v);
    B.defocus = c.defocus_angle > 0 ? 1 : 0;
    auto putd = [](double* dst, D3 s) { dst[0] = s.x; dst[1] = s.y; dst[2] = s.z; };
    putd(B.d.center, lookfrom);
    putd(B.d.dir00, dir00);
    putd(B.d.du, du);
    putd(B.d.dv, dv);
    return B;
}

// copies the camera fields of a CameraBlock into a DevScene or a ViewRecord
template <class Cam>
static void put_camera(Cam& dst, const CameraBlock& B) {
    std::memcpy(dst.center, B.center, sizeof B.center);
    std::memcpy(dst.dir00, B.dir00, sizeof B.dir00);
    std::memcpy(dst.du, B.du, sizeof B.du);
    std::memcpy(dst.dv, B.dv, sizeof B.dv);
    std::memcpy(dst.disk_u, B.disk_u, sizeof B.disk_u);
    std::memcpy(dst.disk_v, B.disk_v, sizeof B.disk_v);
    dst.defocus = B.defocus;
}

static void put_background(DevScene& S, const rt_camera& c) {
    for (int k = 0; k < 3; k++) S.background[k] = (float)c.background[k];
}

// the uploaded camera's block for a width x height frame, into the scene the kernels get
static void setup_camera(DevCtx* ctx, int width, int height) {
    const CameraBlock B = camera_block(ctx->camera, width, height);
    put_camera(ctx->scene, B);
    put_background(ctx->scene, ctx->camera);
    ctx->camera_d = B.d;
    ctx->cam_w = width;
    ctx->cam_h = height;
}

// `too_deep` is set when the device-built tree is deeper than the traversal stack allows; the
// caller then repeats the upload on the host path.
// Are these six baked primitives the faces of ONE parallelepiped (box() of quad.h:76-97 under any rigid transform)?
// Then the boundary is the intersection of three slabs {axis_k, lo_k, hi_k} (boundary_pair_box, rt_device.cuh).
// Checked, not assumed: three pairs of parallel quads, independent axes, and every corner of every quad on a boundary
// plane of each of the other two slabs, with both planes of each reached (the quad IS the whole face).
static bool box_slabs(const rtprep::BakedPrim* q, float4 out[4]) {
    using rtprep::D3;
    D3 n[6];
    double dq[6], scale = 0.0;
    for (int i = 0; i < 6; i++) {
        if (q[i].dev_type != PT_QUAD) return false;
        const D3 c = rtprep::dcross(q[i].b, q[i].c);
        const double len = std::sqrt(rtprep::ddot(c, c));
        if (!(len > 0.0)) return false;
        n[i] = (1.0 / len) * c;
        dq[i] = rtprep::ddot(n[i], q[i].a);
        scale = std::max({scale, std::fabs(dq[i]), std::sqrt(rtprep::ddot(q[i].b, q[i].b)), std::sqrt(rtprep::ddot(q[i].c, q[i].c))});
    }
    const double tol = 1e-9 * std::max(scale, 1.0);
    int mate[6] = {-1, -1, -1, -1, -1, -1}, axis_of[6], n_axes = 0;
    D3 axis[3];
    double lo[3], hi[3];
    for (int i = 0; i < 6; i++) {
        if (mate[i] >= 0) continue;
        for (int j = i + 1; j < 6; j++)
            if (mate[j] < 0 && std::fabs(std::fabs(rtprep::ddot(n[i], n[j])) - 1.0) < 1e-12) { mate[i] = j; mate[j] = i; break; }
        if (mate[i] < 0 || n_axes == 3) return false;
        const int j = mate[i];
        const double dj = rtprep::ddot(n[i], q[j].a);  // the mate's plane along THIS normal
        axis[n_axes] = n[i];
        lo[n_axes] = std::min(dq[i], dj);
        hi[n_axes] = std::max(dq[i], dj);
        if (!(hi[n_axes] - lo[n_axes] > tol)) return false;
        axis_of[i] = axis_of[j] = n_axes++;
    }
    if (n_axes != 3) return false;
    if (!(std::fabs(rtprep::ddot(axis[0], rtprep::dcross(axis[1], axis[2]))) > 1e-6)) return false;
    for (int i = 0; i < 6; i++) {
        const D3 corner[4] = {q[i].a, q[i].a + q[i].b, q[i].a + q[i].c, q[i].a + q[i].b + q[i].c};
        for (int k = 0; k < 3; k++) {
            bool at_lo = false, at_hi = false;
            for (const D3& p : corner) {
                const double v = rtprep::ddot(axis[k], p);
                const bool l = std::fabs(v - lo[k]) <= tol, h = std::fabs(v - hi[k]) <= tol;
                if (!l && !h) return false;
                at_lo |= l;
                at_hi |= h;
            }
            if (k == axis_of[i] ? (at_lo && at_hi) : !(at_lo && at_hi)) return false;  // own axis: one plane; others: both
        }
    }
    for (int k = 0; k < 3; k++) out[k] = make_float4((float)axis[k].x, (float)axis[k].y, (float)axis[k].z, (float)lo[k]);
    out[3] = make_float4((float)hi[0], (float)hi[1], (float)hi[2], 0.0f);
    return true;
}

// The device records the host emits, in the typed arrays of the arena, after `base[t]` records of each type: the host
// path emits the world primitives in leaf order and then the boundaries from base 0; the device path and
// rt_refit_scene emit the boundaries only, after the world records the kernels write.
struct TypedRecords {
    size_t base[4] = {0, 0, 0, 0};
    std::vector<float4> sph, msph, quad, tri, tri_sh;
    std::vector<double> sph_d, msph_d, quad_d, tri_d;
    std::vector<int4> sph_sh, msph_sh, quad_sh;
    // appends the record of `b`; returns its packed ref type << 28 | index
    uint32_t emit(const BakedPrim& b) {
        auto f4 = [](rtprep::F4 v) { return make_float4(v.x, v.y, v.z, v.w); };
        auto i4 = [](rtprep::I4 v) { return make_int4(v.x, v.y, v.z, v.w); };
        if (b.dev_type == PT_SPHERE) {
            const rtprep::SphereRec r = rtprep::make_sphere(b);
            sph.push_back(f4(r.g));
            sph_d.insert(sph_d.end(), r.d, r.d + 4);
            sph_sh.push_back(i4(r.sh));
            return (PT_SPHERE << 28) | (uint32_t)(base[PT_SPHERE] + sph.size() - 1);
        } else if (b.dev_type == PT_MSPHERE) {
            const rtprep::MSphereRec r = rtprep::make_msphere(b);
            msph.push_back(f4(r.g0));
            msph.push_back(f4(r.g1));
            msph_d.insert(msph_d.end(), r.d, r.d + 8);
            msph_sh.push_back(i4(r.sh));
            return (PT_MSPHERE << 28) | (uint32_t)(base[PT_MSPHERE] + msph_sh.size() - 1);
        } else if (b.dev_type == PT_QUAD) {
            const rtprep::QuadRec r = rtprep::make_quad(b);
            for (int k = 0; k < 3; k++) quad.push_back(f4(r.q[k]));
            quad_d.insert(quad_d.end(), r.d, r.d + 12);
            quad_sh.push_back(i4(r.sh));
            return (PT_QUAD << 28) | (uint32_t)(base[PT_QUAD] + quad_sh.size() - 1);
        } else {
            const rtprep::TriRec r = rtprep::make_triangle(b);
            for (int k = 0; k < 3; k++) tri.push_back(f4(r.t[k]));
            tri_d.insert(tri_d.end(), r.d, r.d + 9);
            for (int k = 0; k < 3; k++) tri_sh.push_back(f4(r.sh[k]));
            return (PT_TRI << 28) | (uint32_t)(base[PT_TRI] + tri_sh.size() / 3 - 1);
        }
    }
};

// A quad with an emissive material and a non-zero area joins the next-event emitter list (RT_FLAG_NEE); `area` is the
// running total, the cdf is normalised by finish_emitters.
static bool add_emitter(const rt_scene_desc* sc, const BakedPrim& b, std::vector<DevNeeLight>& lights, double& area_sum) {
    if (b.dev_type != PT_QUAD || b.material < 0 || b.material >= sc->n_materials) return false;
    const rt_material& m = sc->materials[b.material];
    if (m.type != RT_MAT_DIFFUSE_LIGHT && m.type != RT_MAT_EMISSIVE_LIGHT) return false;
    const D3 nn = dcross(b.b, b.c);
    const double area = std::sqrt(ddot(nn, nn));
    if (!(area > 0.0)) return false;
    DevNeeLight lt;
    std::memset(&lt, 0, sizeof lt);
    lt.Q[0] = (float)b.a.x; lt.Q[1] = (float)b.a.y; lt.Q[2] = (float)b.a.z;
    lt.u[0] = (float)b.b.x; lt.u[1] = (float)b.b.y; lt.u[2] = (float)b.b.z;
    lt.v[0] = (float)b.c.x; lt.v[1] = (float)b.c.y; lt.v[2] = (float)b.c.z;
    lt.n[0] = (float)(nn.x / area); lt.n[1] = (float)(nn.y / area); lt.n[2] = (float)(nn.z / area);
    lt.area = (float)area;
    lt.tex = m.texture;
    area_sum += area;
    lt.cdf = (float)area_sum;
    lights.push_back(lt);
    return true;
}
static void finish_emitters(std::vector<DevNeeLight>& lights, double area_sum) {
    for (DevNeeLight& lt : lights) lt.cdf = (float)(lt.cdf / area_sum);
    if (!lights.empty()) lights.back().cdf = 1.0f;
}

// which boundary class a medium has: 1 one sphere, 2 a six-quad box (box_slabs), 0 general
static int8_t media_class(const DevMedium& d) { return d.sphere >= 0 ? 1 : (d.box >= 0 ? 2 : 0); }

// The scene's tables as the render kernels read them.  `boundaries` are the baked boundary primitives and
// `boundary_packed` their records; the image table's texel pointers are left null.
struct SceneTables {
    std::vector<DevMaterial> mats;
    std::vector<DevTexture> texs;
    std::vector<DevImage> images;
    std::vector<float4> perlin_vec;
    std::vector<unsigned char> perlin_perm;
    std::vector<DevMedium> media;
    std::vector<float4> media_box;
    std::vector<DevLight> lights;
    std::vector<float> xrot;
};
static void derive_tables(const rt_scene_desc* sc, const BakedPrim* boundaries, const std::vector<uint32_t>& boundary_packed, SceneTables& T) {
    std::vector<DevMaterial>& mats = T.mats;
    mats.resize((size_t)sc->n_materials);
    for (int i = 0; i < sc->n_materials; i++) {
        const rt_material& m = sc->materials[i];
        DevMaterial& d = mats[i];
        d.type = m.type;
        d.tex = m.texture;
        for (int k = 0; k < 3; k++) d.albedo[k] = (float)m.albedo[k];
        d.param = (float)m.param;
        d.needs_uv = texture_needs_uv(sc, m.texture) ? 1 : 0;
        d.pad = 0;
    }
    std::vector<DevTexture>& texs = T.texs;
    texs.resize((size_t)sc->n_textures);
    for (int i = 0; i < sc->n_textures; i++) {
        const rt_texture& t = sc->textures[i];
        DevTexture& d = texs[i];
        d.type = t.type;
        d.a = t.type == RT_TEX_IMAGE ? t.image : (t.type == RT_TEX_NOISE ? t.perlin : t.even);
        d.b = t.odd;
        d.scale = (float)t.scale;
        for (int k = 0; k < 3; k++) d.color[k] = (float)t.color[k];
        d.pad = 0;
    }
    std::vector<DevImage>& images = T.images;
    images.resize((size_t)sc->n_images);
    for (int i = 0; i < sc->n_images; i++) {
        images[i].rgb = nullptr;
        images[i].w = sc->images[i].width;
        images[i].h = sc->images[i].height;
    }
    std::vector<float4>& perlin_vec = T.perlin_vec;
    std::vector<unsigned char>& perlin_perm = T.perlin_perm;
    perlin_vec.resize((size_t)sc->n_perlins * 256);
    perlin_perm.resize((size_t)sc->n_perlins * 768);
    for (int i = 0; i < sc->n_perlins; i++) {
        const rt_perlin& p = sc->perlins[i];
        for (int k = 0; k < 256; k++) {
            perlin_vec[(size_t)i * 256 + k] = make_float4((float)p.randvec[k][0], (float)p.randvec[k][1], (float)p.randvec[k][2], 0.0f);
            perlin_perm[(size_t)i * 768 + k] = (unsigned char)p.perm_x[k];
            perlin_perm[(size_t)i * 768 + 256 + k] = (unsigned char)p.perm_y[k];
            perlin_perm[(size_t)i * 768 + 512 + k] = (unsigned char)p.perm_z[k];
        }
    }
    std::vector<DevMedium>& media = T.media;
    std::vector<float4>& media_box = T.media_box;
    media.resize((size_t)sc->n_media);
    for (int i = 0; i < sc->n_media; i++) {
        const rt_medium& m = sc->media[i];
        DevMedium& d = media[i];
        std::memset(&d, 0, sizeof d);
        d.bfirst = m.boundary_first;
        d.bcount = m.boundary_count;
        d.neg_inv_density = (float)(-1.0 / (m.density * m.multiplicity));
        d.material = m.material;
        D3 n = xf_dir(m.xform >= 0 ? &sc->xforms[m.xform] : nullptr, D3{1, 0, 0});
        d.normal[0] = (float)n.x; d.normal[1] = (float)n.y; d.normal[2] = (float)n.z;
        d.sphere = -1;
        d.box = -1;
        if (m.boundary_count == 1 && (boundary_packed[m.boundary_first] >> 28) == PT_SPHERE)
            d.sphere = (int)(boundary_packed[m.boundary_first] & 0x0fffffffu);
        float4 slabs[4];
        if (m.boundary_count == 6 && !getenv("RT_B200_NO_BOX_MEDIA") && box_slabs(boundaries + m.boundary_first, slabs)) {
            d.box = (int)(media_box.size() / 4);
            media_box.insert(media_box.end(), slabs, slabs + 4);
        }
    }
    std::vector<DevLight>& lights = T.lights;
    lights.resize((size_t)sc->n_lights);
    for (int i = 0; i < sc->n_lights; i++) {
        const rt_point_light& l = sc->lights[i];
        for (int k = 0; k < 3; k++) { lights[i].pos[k] = (float)l.position[k]; lights[i].intensity[k] = (float)l.intensity[k]; }
        lights[i].size = (float)l.size;
        lights[i].pad = 0;
    }
    std::vector<float>& xrot = T.xrot;
    xrot.resize((size_t)sc->n_xforms * 9);
    for (int i = 0; i < sc->n_xforms; i++)
        for (int k = 0; k < 9; k++) xrot[(size_t)i * 9 + k] = (float)sc->xforms[i].r[k];
}

// FEAT_* bits and the LITE conditions of a scene: `msph` / `tri`: it has moving spheres / triangles
static void set_features(DevCtx* ctx, const rt_scene_desc* sc, const std::vector<DevMedium>& media, bool msph, bool tri) {
    ctx->scene_feat = 0;
    if (sc->n_media > 0) ctx->scene_feat |= FEAT_MEDIA;
    for (const DevMedium& d : media)
        if (d.sphere < 0) ctx->scene_feat |= FEAT_MEDIA_GENERAL;
    for (int i = 0; i < sc->n_materials; i++)
        if (sc->materials[i].type == RT_MAT_SPECULAR) ctx->scene_feat |= FEAT_SPECULAR;
    if (msph) ctx->scene_feat |= FEAT_MSPHERE;
    if (tri) ctx->scene_feat |= FEAT_TRI;
    if (sc->n_lights > 0) ctx->scene_feat |= FEAT_LIGHTS;
    if (sc->camera.defocus_angle > 0) ctx->scene_feat |= FEAT_DEFOCUS;
    ctx->geom_lite = !tri && sc->n_lights == 0;
    ctx->scene_lite = ctx->geom_lite && !(sc->camera.defocus_angle > 0);
}

// the work space of the device build and of rt_refit_scene, grown to `bytes`
static int ensure_scratch(DevCtx* ctx, size_t bytes, const char* entry) {
    if (bytes <= ctx->scratch_cap) return RT_OK;
    if (ctx->scratch) cudaFree(ctx->scratch);
    ctx->scratch = nullptr;
    ctx->scratch_cap = 0;
    size_t cap = bytes + bytes / 8;
    if (cudaMalloc(&ctx->scratch, cap) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "%s: cannot allocate %zu bytes of build work space", entry, cap);
    ctx->scratch_cap = cap;
    return RT_OK;
}

static int upload_scene_impl(DevCtx* ctx, const rt_scene_desc* sc, bool device_build, bool* too_deep) {
    auto t_begin = std::chrono::steady_clock::now();
    int rc;
    const rtprep::Sources src{sc->spheres, sc->quads, sc->triangles, sc->xforms, sc->meshes};
    const int n_prims = ctx->n_prims;      // the world list with every mesh ref expanded: canonical ids 0 .. n_prims - 1
    size_t world_count[4] = {0, 0, 0, 0};  // device path: primitives of each device type the kernels will write

    // ---- bake instance transforms, build per-primitive bounds -----------------------
    std::vector<BakedPrim> baked;
    rtbvh::Result bvh;
    if (device_build) {
        for (int k = 0; k < 4; k++) world_count[k] = ctx->world_type_count[k];
        baked.reserve((size_t)sc->n_boundary_refs);
        for (int i = 0; i < sc->n_boundary_refs; i++) baked.push_back(rtprep::bake_prim(src, sc->boundary_refs[i], -1));
    } else {
        for (int k = 0; k < 4; k++) world_count[k] = 0;
        baked.reserve((size_t)n_prims + sc->n_boundary_refs);
        for (int i = 0; i < sc->n_world; i++) {
            const rt_prim_ref r = sc->world[i];
            if (r.type != RT_PRIM_MESH) {
                baked.push_back(rtprep::bake_prim(src, r, (int)baked.size()));
                continue;
            }
            for (int k = 0; k < sc->meshes[r.index].n_triangles; k++) baked.push_back(rtprep::bake_mesh_triangle(src, r.index, (uint32_t)k, (int)baked.size()));
        }
        for (int i = 0; i < sc->n_boundary_refs; i++) baked.push_back(rtprep::bake_prim(src, sc->boundary_refs[i], -1));

        std::vector<rtbvh::Prim> prims((size_t)n_prims);
        for (int i = 0; i < n_prims; i++) {
            rtbvh::Prim& p = prims[i];
            rtprep::prim_bounds(baked[i], p.box.lo, p.box.hi);
            for (int k = 0; k < 3; k++) p.centroid[k] = 0.5f * (p.box.lo[k] + p.box.hi[k]);
            p.type = baked[i].dev_type;
            p.index = (uint32_t)i;
            p.cost = baked[i].dev_type == PT_SPHERE ? 1.0f : (baked[i].dev_type == PT_MSPHERE ? 1.2f : 1.3f);
        }
        rtbvh::build_bvh(prims, bvh);
    }
    const size_t first_boundary = device_build ? 0 : (size_t)n_prims;

    // ---- device arrays in leaf order, boundaries appended ------------------------------
    TypedRecords recs;
    for (int k = 0; k < 4; k++) recs.base[k] = world_count[k];
    std::vector<uint32_t> boundary_packed((size_t)sc->n_boundary_refs);
    // quads with an emissive material are also listed for the opt-in next-event estimation
    std::vector<DevNeeLight> nee_lights;
    std::vector<int32_t> nee_ids;
    double nee_area = 0.0;
    for (uint32_t id : bvh.order) {
        const BakedPrim& b = baked[id];
        const uint32_t packed = recs.emit(b);
        if (!add_emitter(sc, b, nee_lights, nee_area)) continue;
        recs.quad_sh[(packed & 0x0fffffffu) - world_count[PT_QUAD]].w = (int)nee_lights.size();
        nee_ids.push_back((int32_t)id);
    }
    // device path: the emitters are found in the source array (one pass over the quads, not over the
    // world list); the kernels that write the quad records look the light number up by source index
    std::vector<int32_t> quad_light;
    if (device_build) {
        // only quads the WORLD list references can be hit, so only those are emitters to sample: a quad that is just
        // the boundary of a medium, or that nothing references, would add radiance the reference does not have
        std::vector<char> in_world((size_t)sc->n_quads, 0);
        for (int i = 0; i < sc->n_world; i++)
            if (sc->world[i].type == RT_PRIM_QUAD) in_world[(size_t)sc->world[i].index] = 1;
        for (int i = 0; i < sc->n_quads; i++) {
            if (!in_world[(size_t)i]) continue;
            if (!add_emitter(sc, rtprep::bake_prim(src, rt_prim_ref{RT_PRIM_QUAD, i}, -1), nee_lights, nee_area)) continue;
            if (quad_light.empty()) quad_light.assign((size_t)sc->n_quads, 0);
            quad_light[(size_t)i] = (int32_t)nee_lights.size();
            nee_ids.push_back(i);
        }
    }
    finish_emitters(nee_lights, nee_area);
    for (int i = 0; i < sc->n_boundary_refs; i++) boundary_packed[i] = recs.emit(baked[first_boundary + i]);

    // ---- tables ---------------------------------------------------------------------------
    SceneTables tables;
    derive_tables(sc, baked.data() + first_boundary, boundary_packed, tables);

    std::vector<float4> nodes(bvh.nodes.size() * 4);
    static_assert(sizeof(rtbvh::Node) == 64, "node layout");
    std::memcpy(nodes.data(), bvh.nodes.data(), bvh.nodes.size() * 64);
    for (size_t i = 0; i < bvh.nodes.size(); i++) pair_node(&nodes[4 * i]);

    // ---- the wide quantised tree, collapsed from the SAH BVH2 (host-built scenes) -----------------
    rtwide::Built wide;
    if (!device_build && ctx->bvh_width != 2 && n_prims > 0) {
        float wlo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, whi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        for (int i = 0; i < n_prims; i++) {
            float lo[3], hi[3];
            rtprep::prim_bounds(baked[i], lo, hi);
            for (int k = 0; k < 3; k++) {
                const float e = 1e-6f * std::max({1.0f, std::fabs(lo[k]), std::fabs(hi[k])});
                wlo[k] = std::min(wlo[k], lo[k] - e);
                whi[k] = std::max(whi[k], hi[k] + e);
            }
        }
        if (ctx->bvh_width == 8) rtwide::build_wide<8>(bvh, true, wlo, whi, wide);
        else rtwide::build_wide<4>(bvh, true, wlo, whi, wide);
        if (wide.depth > (uint32_t)kWideMaxDepth) wide = rtwide::Built();  // degenerate tree: keep the binary one
    }

    DevScene& S = ctx->scene;
    std::memset(&S, 0, sizeof S);
    // ---- one arena.  Host path: everything is staged in pinned memory at its arena offset and moved
    // with ONE copy.  Device path: the typed arrays and the nodes are written by kernels (`skip` bytes
    // at the front of a block: the world primitives), only the tables and the boundary records that
    // follow the world primitives are staged, compactly, and copied block by block.
    ArenaPlan plan, stage;
    std::vector<size_t> img_off((size_t)sc->n_images), img_stage((size_t)sc->n_images);
    for (int i = 0; i < sc->n_images; i++) {
        img_off[i] = plan.add((size_t)sc->images[i].width * sc->images[i].height * 3);
        img_stage[i] = stage.add((size_t)sc->images[i].width * sc->images[i].height * 3);
    }
    struct Block { const void* src; size_t bytes, off, skip, stage_off; const void** field; };
    std::vector<Block> blocks;
    auto add_block = [&](const void* data, size_t bytes, size_t skip, const void** field) {
        Block b{data, bytes, plan.add(skip + bytes), skip, 0, field};
        b.stage_off = stage.add(bytes);
        blocks.push_back(b);
    };
    // device path: n - 1 radix-tree slots + room for the SAH top tree over at most kMaxClusters clusters
    const size_t node_skip = device_build ? ((size_t)(n_prims - 1) + rtlbvh::kMaxClusters) * 64 : 0;
#define UP(vec, field) add_block(vec.data(), vec.size() * sizeof(vec[0]), 0, (const void**)&S.field);
#define UPW(vec, field, type, rec_bytes) add_block(recs.vec.data(), recs.vec.size() * sizeof(recs.vec[0]), world_count[type] * (size_t)(rec_bytes), (const void**)&S.field);
    add_block(nodes.data(), device_build ? 0 : nodes.size() * sizeof(float4), node_skip, (const void**)&S.nodes);
    if (wide.n_nodes) {
        add_block(wide.words.data(), wide.words.size() * sizeof(uint32_t), 0, (const void**)&S.wnodes);
        add_block(wide.refs.data(), wide.refs.size() * sizeof(int32_t), 0, (const void**)&S.wrefs);
    }
    UPW(sph, sph, PT_SPHERE, 16) UPW(msph, msph, PT_MSPHERE, 32) UPW(quad, quad, PT_QUAD, 48) UPW(tri, tri, PT_TRI, 48)
    UPW(sph_d, sph_d, PT_SPHERE, 32) UPW(msph_d, msph_d, PT_MSPHERE, 64) UPW(quad_d, quad_d, PT_QUAD, 96) UPW(tri_d, tri_d, PT_TRI, 72)
    UPW(sph_sh, sph_sh, PT_SPHERE, 16) UPW(msph_sh, msph_sh, PT_MSPHERE, 16) UPW(quad_sh, quad_sh, PT_QUAD, 16) UPW(tri_sh, tri_sh, PT_TRI, 48)
    UP(tables.xrot, xrot) UP(tables.media, media) UP(tables.media_box, media_box)
    UP(boundary_packed, boundary) UP(tables.mats, mats) UP(tables.texs, texs) UP(tables.images, images) UP(tables.perlin_vec, perlin_vec)
    UP(tables.perlin_perm, perlin_perm) UP(tables.lights, lights) UP(nee_lights, nee_lights)
#undef UP
#undef UPW
    if (plan.size > ctx->arena_cap) {
        if (ctx->arena) cudaFree(ctx->arena);
        ctx->arena = nullptr;
        ctx->arena_cap = 0;
        size_t cap = plan.size + plan.size / 4;
        if (cudaMalloc(&ctx->arena, cap) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "rt_upload_scene: cannot allocate %zu bytes of device memory", cap);
        ctx->arena_cap = cap;
    }
    const size_t stage_need = device_build ? stage.size : plan.size;
    if (stage_need > ctx->staging_cap) {
        if (ctx->staging) cudaFreeHost(ctx->staging);
        ctx->staging = nullptr;
        ctx->staging_cap = 0;
        size_t cap = stage_need + stage_need / 4;
        if (cudaHostAlloc(&ctx->staging, cap, cudaHostAllocDefault) != cudaSuccess)
            return fail(ctx, RT_ERR_NOMEM, "rt_upload_scene: cannot allocate %zu bytes of pinned host memory", cap);
        ctx->staging_cap = cap;
    }
    for (int i = 0; i < sc->n_images; i++) {
        tables.images[i].rgb = ctx->arena + img_off[i];
        std::memcpy(ctx->staging + (device_build ? img_stage[i] : img_off[i]), sc->images[i].rgb, (size_t)sc->images[i].width * sc->images[i].height * 3);
    }
    for (const Block& b : blocks) {
        if (b.bytes) std::memcpy(ctx->staging + (device_build ? b.stage_off : b.off), b.src, b.bytes);
        *b.field = ctx->arena + b.off;
    }
    // the traversal stack is not bounds-checked on the device (rt_device.cuh, Trav::interior)
    if (!device_build && bvh.depth >= (uint32_t)STACK_SIZE)
        return fail(ctx, RT_ERR_UNSUPPORTED, "rt_upload_scene: the BVH has %u levels, the traversal stack holds %d", bvh.depth, STACK_SIZE);
    uint32_t n_nodes = (uint32_t)bvh.nodes.size(), depth = bvh.depth, leaves = bvh.leaves;
    int root = bvh.root, device_nodes = 0;
    if (!device_build) {
        CU(ctx, cudaMemcpyAsync(ctx->arena, ctx->staging, plan.size, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->staged_bytes = plan.size;
        ctx->stats.upload_bytes = plan.size;
    } else {
        size_t staged = 0;
        for (int i = 0; i < sc->n_images; i++) {
            const size_t bytes = (size_t)sc->images[i].width * sc->images[i].height * 3;
            CU(ctx, cudaMemcpyAsync(ctx->arena + img_off[i], ctx->staging + img_stage[i], bytes, cudaMemcpyHostToDevice, ctx->stream));
            staged += bytes;
        }
        for (const Block& b : blocks)
            if (b.bytes) {
                CU(ctx, cudaMemcpyAsync(ctx->arena + b.off + b.skip, ctx->staging + b.stage_off, b.bytes, cudaMemcpyHostToDevice, ctx->stream));
                staged += b.bytes;
            }
        const rtlbvh::Layout L = rtlbvh::plan_scratch(sc, n_prims);
        if ((rc = ensure_scratch(ctx, L.total, "rt_upload_scene")) != RT_OK) return rc;
        rtlbvh::Targets T;
        T.nodes = (float4*)S.nodes;
        T.sph = (float4*)S.sph; T.msph = (float4*)S.msph; T.quad = (float4*)S.quad; T.tri = (float4*)S.tri; T.tri_sh = (float4*)S.tri_sh;
        T.sph_d = (double*)S.sph_d; T.msph_d = (double*)S.msph_d; T.quad_d = (double*)S.quad_d; T.tri_d = (double*)S.tri_d;
        T.sph_sh = (int4*)S.sph_sh; T.msph_sh = (int4*)S.msph_sh; T.quad_sh = (int4*)S.quad_sh;
        rtlbvh::BuildResult br;
        if (L.largest_input >= 4 * rtlbvh::kCopyChunk) CU(ctx, ctx->copy_ring.init());
        CU(ctx, rtlbvh::build_on_device(sc, n_prims, ctx->scratch, L, T, ctx->stream, ctx->copy_ring, ctx->device, ctx->bvh_builder != 3,
                                        quad_light.empty() ? nullptr : quad_light.data(), br));
        n_nodes = br.nodes;
        depth = br.depth;
        leaves = br.leaves;
        root = br.root;
        device_nodes = n_prims - 1 + (int)br.top_nodes;
        // what crossed to the device: the raw arrays (and top levels) plus the staged tables and images
        ctx->stats.upload_bytes = br.bytes_in + staged;
        ctx->stats.device_build_ms = br.ms_build + br.ms_emit;
        ctx->stats.device_top_ms = br.ms_top;
        ctx->stats.device_copy_in_ms = br.ms_copy_in;
        if (depth >= (uint32_t)STACK_SIZE - 2) {
            *too_deep = true;
            return RT_OK;
        }
        if (device_nodes > 0) {
            pair_nodes_kernel<<<(device_nodes + 255) / 256, 256, 0, ctx->stream>>>((float4*)S.nodes, device_nodes);
            CU(ctx, cudaGetLastError());
            CU(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    ctx->stats.bvh_on_device = device_build ? 1 : 0;
    S.root = root;
    S.n_nodes = device_build ? device_nodes : (int)bvh.nodes.size();
    S.n_world = n_prims;
    S.n_media = sc->n_media;
    S.n_lights = sc->n_lights;
    S.n_nee_lights = (int)nee_lights.size();
    S.nee_total_area = (float)nee_area;
    S.wide_width = wide.n_nodes ? wide.width : 0;
    S.f32_one_bits = 0x3F800000u;
    if (!wide.n_nodes) { S.wnodes = nullptr; S.wrefs = nullptr; }
    ctx->wide_depth = (int)wide.depth;
    ctx->stats.bvh_width = wide.n_nodes ? (uint32_t)wide.width : 2u;
    ctx->stats.wide_nodes = wide.n_nodes;
    ctx->stats.wide_depth = wide.depth;
    ctx->camera = sc->camera;
    ctx->n_materials = sc->n_materials;
    ctx->n_textures = sc->n_textures;
    set_features(ctx, sc, tables.media, world_count[PT_MSPHERE] > 0 || !recs.msph.empty(), !recs.tri.empty() || world_count[PT_TRI] > 0);
    ctx->cam_w = ctx->cam_h = 0;
    ctx->has_scene = true;
    // the structure rt_refit_scene holds a description to
    DevCtx::Shape& sh = ctx->shape;
    const int32_t counts[13] = {sc->n_world, sc->n_boundary_refs, sc->n_spheres, sc->n_quads, sc->n_triangles, sc->n_media, sc->n_xforms,
                                sc->n_materials, sc->n_textures, sc->n_images, sc->n_perlins, sc->n_lights, sc->n_meshes};
    std::memcpy(sh.counts, counts, sizeof counts);
    sh.mesh_tris.clear();
    for (int i = 0; i < sc->n_meshes; i++) sh.mesh_tris.push_back(sc->meshes[i].n_triangles);
    sh.image_wh.clear();
    sh.image_dev.clear();
    for (int i = 0; i < sc->n_images; i++) {
        sh.image_wh.push_back(sc->images[i].width);
        sh.image_wh.push_back(sc->images[i].height);
        sh.image_dev.push_back(ctx->arena + img_off[i]);
    }
    sh.boundary_packed = boundary_packed;
    sh.media_class.clear();
    for (const DevMedium& d : tables.media) sh.media_class.push_back(media_class(d));
    sh.nee_ids = nee_ids;
    sh.n_prims = n_prims;
    sh.device_built = device_build;
    for (int k = 0; k < 4; k++) sh.world_type_count[k] = ctx->world_type_count[k];
    ctx->refit_tree.levels.clear();
    ctx->stats.bvh_nodes = n_nodes;
    ctx->stats.bvh_depth = depth;
    ctx->stats.bvh_leaves = leaves;
    ctx->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return RT_OK;
}

static int dev_wait(DevCtx* ctx);

static int dev_upload_scene(DevCtx* ctx, const rt_scene_desc* sc) {
    if (!ctx) return RT_ERR_INVALID;
    auto t_begin = std::chrono::steady_clock::now();
    int rc = validate_scene(ctx, sc, /*shallow=*/true);
    if (rc != RT_OK) return rc;
    CU(ctx, cudaSetDevice(ctx->device));
    // an asynchronous render may still be reading the arena -- on the caller's stream, not necessarily ours
    rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    // which path: host (bake + binned SAH on the CPU) or device (csrc/bvh_device.cuh)
    const int n_prims = ctx->n_prims;
    const bool device_build = n_prims >= kDeviceBuildMin && (ctx->bvh_builder >= 2 || (ctx->bvh_builder == 0 && n_prims >= kDeviceBuildAuto));
    // the same scene again (same bytes, same builder settings): the staged arena is still in pinned memory -- copy it, done.
    // Only the host path leaves its whole arena staged, so only a host-path scene is fingerprinted (hashing a
    // device-path scene would cost more than its upload)
    const bool cache = !getenv("RT_B200_NO_SCENE_CACHE");
    uint64_t key = cache && !device_build ? scene_key(ctx, sc) : 0;
    if (key && ctx->has_scene && ctx->staged_key == key && ctx->staged_bytes > 0) {
        CU(ctx, cudaMemcpyAsync(ctx->arena, ctx->staging, ctx->staged_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        const DevCtx::SceneState& st = ctx->staged_state;
        ctx->scene = st.scene;
        ctx->camera = st.camera;
        ctx->scene_feat = st.scene_feat;
        ctx->scene_lite = st.scene_lite;
        ctx->geom_lite = st.geom_lite;
        ctx->cam_w = ctx->cam_h = 0;
        ctx->stats.scene_reused = 1;
        ctx->stats.upload_bytes = ctx->staged_bytes;
        ctx->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        return RT_OK;
    }
    ctx->staged_key = 0;
    ctx->staged_bytes = 0;
    ctx->stats.scene_reused = 0;
    rc = validate_scene(ctx, sc, /*shallow=*/false);
    if (rc != RT_OK) return rc;
    free_scene(ctx);
    ctx->stats.device_build_ms = ctx->stats.device_copy_in_ms = ctx->stats.device_top_ms = 0;
    bool too_deep = false;
    rc = upload_scene_impl(ctx, sc, device_build, &too_deep);
    if (rc == RT_OK && too_deep) {
        rc = upload_scene_impl(ctx, sc, false, &too_deep);  // degenerate input: the SAH tree is shallow
        if (cache) key = scene_key(ctx, sc);
    }
    if (rc == RT_OK && ctx->staged_bytes > 0) {  // host path: the whole arena sits in the pinned staging buffer
        ctx->staged_key = key;
        ctx->staged_state = DevCtx::SceneState{ctx->scene, ctx->camera, ctx->scene_feat, ctx->scene_lite, ctx->geom_lite};
    }
    if (rc == RT_OK) ctx->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return rc;
}

// rt_refit_scene (bvh_refit.cuh): `sc` has the structure of the uploaded scene; its records, boxes and tables replace
// the uploaded ones, the tree keeps its topology and leaf order.  Everything is checked before the arena is written:
// a refused refit leaves the uploaded scene as it was.
static int dev_refit_scene(DevCtx* ctx, const rt_scene_desc* sc) {
    if (!ctx) return RT_ERR_INVALID;
    auto t_begin = std::chrono::steady_clock::now();
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_refit_scene: no scene uploaded (rt_upload_scene first)");
    DevScene& S = ctx->scene;
    if (S.wide_width)
        return fail(ctx, RT_ERR_UNSUPPORTED, "rt_refit_scene: the uploaded scene is traversed as a %d-wide tree; only the binary tree "
                    "is refitted (rt_set_bvh_width(2) and rt_upload_scene)", S.wide_width);
    // validated like an upload; the counts validate_scene leaves in ctx are the new description's, the uploaded
    // scene's are kept with its structure
    const DevCtx::Shape& sh = ctx->shape;
    const int n_prims = sh.n_prims;
    const size_t* type_count = sh.world_type_count;
    size_t new_count[4];
    int rc = validate_scene(ctx, sc, /*shallow=*/false);
    const int new_prims = ctx->n_prims;
    std::memcpy(new_count, ctx->world_type_count, sizeof new_count);
    if (rc != RT_OK) {
        if (ctx->error.rfind("rt_upload_scene", 0) == 0) ctx->error.replace(0, 15, "rt_refit_scene");
        return rc;
    }
    // ---- the structure, on the host: counts, meshes, images, boundaries, emitters, media -----------------
    static const char* kHint = "; a scene of another structure needs rt_upload_scene";
    static const char* kKind[4] = {"sphere", "moving sphere", "quad", "triangle"};
    static const char* kCountName[13] = {"n_world", "n_boundary_refs", "n_spheres", "n_quads", "n_triangles", "n_media", "n_xforms",
                                         "n_materials", "n_textures", "n_images", "n_perlins", "n_lights", "n_meshes"};
    const int32_t counts[13] = {sc->n_world, sc->n_boundary_refs, sc->n_spheres, sc->n_quads, sc->n_triangles, sc->n_media, sc->n_xforms,
                                sc->n_materials, sc->n_textures, sc->n_images, sc->n_perlins, sc->n_lights, sc->n_meshes};
    for (int k = 0; k < 13; k++)
        if (counts[k] != sh.counts[k])
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: %s is %d, the uploaded scene's %d%s", kCountName[k], counts[k], sh.counts[k], kHint);
    for (int i = 0; i < sc->n_meshes; i++)
        if (sc->meshes[i].n_triangles != sh.mesh_tris[(size_t)i])
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: meshes[%d] has %d triangles, the uploaded scene's %d%s", i, sc->meshes[i].n_triangles,
                        sh.mesh_tris[(size_t)i], kHint);
    for (int i = 0; i < sc->n_images; i++)
        if (sc->images[i].width != sh.image_wh[2 * (size_t)i] || sc->images[i].height != sh.image_wh[2 * (size_t)i + 1])
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: images[%d] is %dx%d, the uploaded scene's %dx%d%s", i, sc->images[i].width,
                        sc->images[i].height, sh.image_wh[2 * (size_t)i], sh.image_wh[2 * (size_t)i + 1], kHint);
    if (new_prims != n_prims)
        return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: the world list has %d primitives, the uploaded scene %d%s", new_prims, n_prims, kHint);
    for (int t = 0; t < 4; t++)
        if (new_count[t] != type_count[t])
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: the world list has %zu primitives of kind %s, the uploaded scene %zu%s", new_count[t],
                        kKind[t], type_count[t], kHint);
    const rtprep::Sources src{sc->spheres, sc->quads, sc->triangles, sc->xforms, sc->meshes};
    std::vector<BakedPrim> boundaries;
    for (int i = 0; i < sc->n_boundary_refs; i++) {
        boundaries.push_back(rtprep::bake_prim(src, sc->boundary_refs[i], -1));
        const uint32_t was = sh.boundary_packed[(size_t)i] >> 28;
        if (boundaries.back().dev_type != was)
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: boundary_refs[%d] changes kind (%s, the uploaded scene's %s)%s", i,
                        kKind[boundaries.back().dev_type], kKind[was], kHint);
    }
    // the emitters of `sc` by the rule of the upload that built the tree, keyed like shape.nee_ids (ascending)
    std::vector<std::pair<int32_t, BakedPrim>> emitters;
    {
        std::vector<DevNeeLight> probe;
        double area = 0.0;
        if (sh.device_built) {
            std::vector<char> in_world((size_t)sc->n_quads, 0);
            for (int i = 0; i < sc->n_world; i++)
                if (sc->world[i].type == RT_PRIM_QUAD) in_world[(size_t)sc->world[i].index] = 1;
            for (int i = 0; i < sc->n_quads; i++) {
                if (!in_world[(size_t)i]) continue;
                const BakedPrim b = rtprep::bake_prim(src, rt_prim_ref{RT_PRIM_QUAD, i}, -1);
                if (add_emitter(sc, b, probe, area)) emitters.emplace_back(i, b);
            }
        } else {
            int32_t id = 0;
            for (int i = 0; i < sc->n_world; i++) {
                const rt_prim_ref r = sc->world[i];
                if (r.type == RT_PRIM_MESH) {
                    id += sc->meshes[r.index].n_triangles;
                    continue;
                }
                if (r.type == RT_PRIM_QUAD) {
                    const BakedPrim b = rtprep::bake_prim(src, r, id);
                    if (add_emitter(sc, b, probe, area)) emitters.emplace_back(id, b);
                }
                id++;
            }
        }
    }
    std::vector<int32_t> listed = sh.nee_ids;
    std::sort(listed.begin(), listed.end());
    for (size_t i = 0; i < std::max(listed.size(), emitters.size()); i++) {
        const int32_t was = i < listed.size() ? listed[i] : INT32_MAX, now = i < emitters.size() ? emitters[i].first : INT32_MAX;
        if (was != now)
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: %s %d %s the next-event emitter list (an emissive material and a non-zero area "
                        "make a quad an emitter)%s", sh.device_built ? "source quad" : "primitive", std::min(was, now),
                        was < now ? "leaves" : "joins", kHint);
    }
    std::vector<DevNeeLight> nee_lights;
    double nee_area = 0.0;
    for (int32_t id : sh.nee_ids) {
        auto it = std::lower_bound(emitters.begin(), emitters.end(), id, [](const std::pair<int32_t, BakedPrim>& e, int32_t v) { return e.first < v; });
        add_emitter(sc, it->second, nee_lights, nee_area);
    }
    finish_emitters(nee_lights, nee_area);
    SceneTables tables;
    derive_tables(sc, boundaries.data(), sh.boundary_packed, tables);
    static const char* kClass[3] = {"general", "one sphere", "a six-quad box"};
    for (int i = 0; i < sc->n_media; i++) {
        const int8_t now = media_class(tables.media[(size_t)i]), was = sh.media_class[(size_t)i];
        if (now != was)
            return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: media[%d] changes its boundary class (%s, the uploaded scene's %s)%s", i, kClass[now],
                        kClass[was], kHint);
    }

    // ---- the inputs on the device, and the kind of every world record slot's primitive -------------------
    CU(ctx, cudaSetDevice(ctx->device));
    const rtlbvh::Layout L = rtlbvh::plan_refit(sc, n_prims);
    if ((rc = ensure_scratch(ctx, L.total, "rt_refit_scene")) != RT_OK) return rc;
    if (L.largest_input >= 4 * rtlbvh::kCopyChunk) CU(ctx, ctx->copy_ring.init());
    size_t bytes_in = 0;
    CU(ctx, rtlbvh::copy_inputs(sc, ctx->scratch, L, ctx->stream, ctx->copy_ring, ctx->device, bytes_in));
    rtlbvh::Scratch W = rtlbvh::input_view(sc, n_prims, ctx->scratch, L);
    W.box_lo = (float4*)(ctx->scratch + L.box_lo);
    W.box_hi = (float4*)(ctx->scratch + L.box_hi);
    W.counters = (unsigned*)(ctx->scratch + L.counters);
    const bool meshes = sc->n_meshes > 0;
    if (meshes && n_prims > 0) CU(ctx, rtlbvh::map_prims(W, sc->n_world, ctx->scratch, L, ctx->scratch + L.cub_temp, L.cub_temp_bytes, ctx->stream));
    rtlbvh::RefitSlots R;
    R.T.nodes = (float4*)S.nodes;
    R.T.sph = (float4*)S.sph; R.T.msph = (float4*)S.msph; R.T.quad = (float4*)S.quad; R.T.tri = (float4*)S.tri; R.T.tri_sh = (float4*)S.tri_sh;
    R.T.sph_d = (double*)S.sph_d; R.T.msph_d = (double*)S.msph_d; R.T.quad_d = (double*)S.quad_d; R.T.tri_d = (double*)S.tri_d;
    R.T.sph_sh = (int4*)S.sph_sh; R.T.msph_sh = (int4*)S.msph_sh; R.T.quad_sh = (int4*)S.quad_sh;
    R.base[0] = 0;
    for (int t = 0; t < 4; t++) R.base[t + 1] = R.base[t] + (unsigned)type_count[t];
    // a device-built tree numbers its emitters by source quad, and a world quad may now name another source quad: the
    // emitter number of each slot follows its quad, as prims_kernel sets it at upload
    R.quad_light = nullptr;
    if (sh.device_built && !sh.nee_ids.empty()) {
        std::vector<int32_t> quad_light((size_t)sc->n_quads, 0);
        for (size_t k = 0; k < sh.nee_ids.size(); k++) quad_light[(size_t)sh.nee_ids[k]] = (int32_t)(k + 1);
        CU(ctx, rtlbvh::copy_in(ctx->scratch + L.quad_light, quad_light.data(), quad_light.size() * sizeof(int32_t), ctx->stream, ctx->copy_ring,
                                ctx->device));
        bytes_in += quad_light.size() * sizeof(int32_t);
        R.quad_light = (const int*)(ctx->scratch + L.quad_light);
    }
    unsigned bad = ~0u;
    if (n_prims > 0) {
        CU(ctx, cudaMemsetAsync(W.counters, 0xff, sizeof bad, ctx->stream));
        if (meshes) rtlbvh::refit_check_kernel<true><<<(n_prims + 255) / 256, 256, 0, ctx->stream>>>(W, R, W.counters);
        else rtlbvh::refit_check_kernel<false><<<(n_prims + 255) / 256, 256, 0, ctx->stream>>>(W, R, W.counters);
        CU(ctx, cudaGetLastError());
        CU(ctx, cudaMemcpyAsync(&bad, W.counters, sizeof bad, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (bad != ~0u)
        return fail(ctx, RT_ERR_INVALID, "rt_refit_scene: world primitive %u changes kind (%s, the uploaded scene's %s)%s", bad >> 4, kKind[bad & 3u],
                    kKind[(bad >> 2) & 3u], kHint);
    // the uploaded tree in breadth-first order, once per upload (n_world == 0: the root is never followed)
    const bool has_tree = S.n_world > 0 && S.root >= 0;
    if (has_tree && ctx->refit_tree.levels.empty()) {
        bool ok = false;
        CU(ctx, rtlbvh::derive_refit_tree(ctx->refit_tree, S.nodes, S.root, S.n_nodes, STACK_SIZE, ctx->sm_count, ctx->stream, ok));
        if (!ok) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_refit_scene: the uploaded tree has more than %d levels", STACK_SIZE);
    }

    // ---- from here on the arena is written: wait for the passes that read it, like an upload ---------------
    rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    CU(ctx, rtlbvh::refit_on_device(W, R, meshes, (float4*)S.nodes, ctx->refit_tree, ctx->stream));
    TypedRecords recs;
    for (int k = 0; k < 4; k++) recs.base[k] = type_count[k];
    for (const BakedPrim& b : boundaries) recs.emit(b);
    auto put = [&](const void* dst, const void* host, size_t bytes) -> cudaError_t {
        if (!bytes) return cudaSuccess;
        bytes_in += bytes;
        return cudaMemcpyAsync((void*)dst, host, bytes, cudaMemcpyHostToDevice, ctx->stream);
    };
#define PUT(vec, field) CU(ctx, put(S.field, vec.data(), vec.size() * sizeof(vec[0])));
#define PUTW(vec, field, type, rec_bytes) \
    CU(ctx, put((const unsigned char*)S.field + type_count[type] * (size_t)(rec_bytes), recs.vec.data(), recs.vec.size() * sizeof(recs.vec[0])));
    PUTW(sph, sph, PT_SPHERE, 16) PUTW(msph, msph, PT_MSPHERE, 32) PUTW(quad, quad, PT_QUAD, 48) PUTW(tri, tri, PT_TRI, 48)
    PUTW(sph_d, sph_d, PT_SPHERE, 32) PUTW(msph_d, msph_d, PT_MSPHERE, 64) PUTW(quad_d, quad_d, PT_QUAD, 96) PUTW(tri_d, tri_d, PT_TRI, 72)
    PUTW(sph_sh, sph_sh, PT_SPHERE, 16) PUTW(msph_sh, msph_sh, PT_MSPHERE, 16) PUTW(quad_sh, quad_sh, PT_QUAD, 16) PUTW(tri_sh, tri_sh, PT_TRI, 48)
    PUT(tables.xrot, xrot) PUT(tables.media, media) PUT(tables.media_box, media_box) PUT(tables.mats, mats) PUT(tables.texs, texs)
    PUT(tables.perlin_vec, perlin_vec) PUT(tables.perlin_perm, perlin_perm) PUT(tables.lights, lights) PUT(nee_lights, nee_lights)
#undef PUT
#undef PUTW
    for (int i = 0; i < sc->n_images; i++) CU(ctx, put(sh.image_dev[(size_t)i], sc->images[i].rgb, (size_t)sc->images[i].width * sc->images[i].height * 3));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    S.nee_total_area = (float)nee_area;
    ctx->camera = sc->camera;
    ctx->cam_w = ctx->cam_h = 0;
    set_features(ctx, sc, tables.media, type_count[PT_MSPHERE] > 0 || !recs.msph.empty(), !recs.tri.empty() || type_count[PT_TRI] > 0);
    ctx->stats.scene_reused = 0;
    ctx->stats.upload_bytes = bytes_in;
    ctx->stats.upload_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return RT_OK;
}

// 0 auto, 1 host SAH, 2 device LBVH: which builder the next rt_upload_scene uses
static int dev_set_bvh_builder(DevCtx* ctx, int32_t mode) {
    if (!ctx) return RT_ERR_INVALID;
    if (mode < 0 || mode > 3) return fail(ctx, RT_ERR_INVALID, "rt_set_bvh_builder: mode %d (0 auto, 1 host, 2 device, 3 device without the SAH top)", mode);
    ctx->bvh_builder = mode;
    return RT_OK;
}

// 2, 4 or 8: which acceleration structure the next rt_upload_scene builds for the render kernels
static int dev_set_bvh_width(DevCtx* ctx, int32_t width) {
    if (!ctx) return RT_ERR_INVALID;
    if (width != 2 && width != 4 && width != 8) return fail(ctx, RT_ERR_INVALID, "rt_set_bvh_width: %d (2 binary, 4 or 8 wide quantised)", width);
    ctx->bvh_width = width;
    return RT_OK;
}

// ---------------------------------------------------------------------------------
// rendering
// ---------------------------------------------------------------------------------
extern "C" size_t rt_shard_pixels(int32_t width, int32_t height, int32_t tile_size, int32_t shard_rank, int32_t shard_count) {
    if (width <= 0 || height <= 0 || tile_size <= 0 || shard_count <= 0 || shard_rank < 0 || shard_rank >= shard_count) return 0;
    AccumLayout L;
    L.width = width; L.height = height; L.compact = true; L.rank = shard_rank; L.count = shard_count; L.tile = tile_size;
    return L.slots();
}

static int ensure_accum(DevCtx* ctx, const AccumLayout& L) {
    const size_t need = std::max<size_t>(L.slots(), 1) * 4 * sizeof(unsigned long long);
    if (ctx->accum_external) {
        if (L.compact || ctx->acc.width != L.width || ctx->acc.height != L.height)
            return fail(ctx, RT_ERR_STATE, "rt_render: the bound accumulation buffer is a full %dx%d frame, this render needs %s%dx%d", ctx->acc.width,
                        ctx->acc.height, L.compact ? "compact tiles of " : "", L.width, L.height);
        return RT_OK;
    }
    if (ctx->accum && ctx->acc == L) return RT_OK;
    ctx->moments_valid = false;
    if (!ctx->accum || need > ctx->accum_cap) {
        if (ctx->accum) cudaFree(ctx->accum);
        ctx->accum = nullptr;
        ctx->accum_cap = 0;
        if (cudaMalloc(&ctx->accum, need) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "rt_render: cannot allocate %zu bytes for the accumulation buffer", need);
        ctx->accum_cap = need;
    }
    ctx->accum_bytes = need;
    ctx->acc = L;
    cudaMemsetAsync(ctx->accum, 0, need, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    return RT_OK;
}

// the moments buffer of RT_FLAG_MOMENTS: 48 bytes per slot, same layout as `accum` (its contents are set by the caller)
static int ensure_moments(DevCtx* ctx, size_t slots) {
    const size_t need = std::max<size_t>(slots, 1) * 6 * sizeof(unsigned long long);
    if (ctx->moments && need <= ctx->moments_cap) return RT_OK;
    if (ctx->moments) cudaFree(ctx->moments);
    ctx->moments = nullptr;
    ctx->moments_cap = 0;
    if (cudaMalloc(&ctx->moments, need) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "cannot allocate %zu bytes for the moments buffer", need);
    ctx->moments_cap = need;
    return RT_OK;
}

static int dev_bind_accum(DevCtx* ctx, void* device_ptr, size_t bytes, int32_t width, int32_t height) {
    if (!ctx) return RT_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    // passes still in flight (asynchronous, overlapped) write into the buffer that is about to be replaced
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    if (ctx->accum && !ctx->accum_external) cudaFree(ctx->accum);
    ctx->accum = nullptr;
    ctx->accum_external = false;
    ctx->acc = AccumLayout();
    ctx->accum_bytes = ctx->accum_cap = 0;
    ctx->moments_valid = ctx->sums_uploaded = false;
    if (!device_ptr) return RT_OK;
    size_t need = (size_t)width * height * 4 * sizeof(unsigned long long);
    if (width <= 0 || height <= 0 || bytes < need) return fail(ctx, RT_ERR_INVALID, "rt_bind_accum: need %zu bytes for %dx%d, got %zu", need, width, height, bytes);
    ctx->accum = (unsigned long long*)device_ptr;
    ctx->accum_external = true;
    ctx->accum_bytes = need;
    ctx->acc.width = width;
    ctx->acc.height = height;
    return RT_OK;
}

static int dev_accum_buffer(DevCtx* ctx, void** device_ptr, size_t* bytes) {
    if (!ctx || !device_ptr || !bytes) return RT_ERR_INVALID;
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "rt_accum_buffer: nothing rendered or bound yet");
    *device_ptr = ctx->accum;
    *bytes = ctx->accum_bytes;
    return RT_OK;
}

// Scatter the compact tile buffers of `count` shards (shard r starts at shards + r * stride bytes) into a full
// row-major frame of `bpp`-byte pixels: pixel (x, y) lies in tile t = (y / tile) * tiles_x + x / tile, which is local
// tile t / count of shard t mod count.  only_rank >= 0: take that shard's tiles from `shards` directly (stride
// unused) and leave the other pixels as they are.  bpp: 3 (RGB8), 12 (float RGB), 32 (the uint64 sums) or 48 (the moments).
template <int BPP>
__global__ void untile_kernel(const unsigned char* __restrict__ shards, size_t stride, int count, int only_rank, int width, int height,
                              int tile, unsigned char* __restrict__ dst) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= width || y >= height) return;
    const int tiles_x = (width + tile - 1) / tile;
    const int t = (y / tile) * tiles_x + x / tile;
    const int r = t % count;
    if (only_rank >= 0 && r != only_rank) return;
    const size_t slot = ((size_t)(t / count) * tile + (size_t)(y % tile)) * tile + (size_t)(x % tile);
    const unsigned char* src = shards + (only_rank >= 0 ? 0 : (size_t)r * stride) + slot * BPP;
    unsigned char* out = dst + ((size_t)y * width + x) * BPP;
    if (BPP == 32) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(out);
        d4[0] = s4[0];
        d4[1] = s4[1];
    } else if (BPP == 12) {
        const float* sf = reinterpret_cast<const float*>(src);
        float* df = reinterpret_cast<float*>(out);
        df[0] = sf[0]; df[1] = sf[1]; df[2] = sf[2];
    } else if (BPP == 48) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(out);
        d4[0] = s4[0];
        d4[1] = s4[1];
        d4[2] = s4[2];
    } else {
        out[0] = src[0]; out[1] = src[1]; out[2] = src[2];
    }
}
// a += b over n uint64 (fixed-point sums are associative: the order of the shards does not matter)
__global__ void add_sums_kernel(unsigned long long* __restrict__ a, const unsigned long long* __restrict__ b, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] += b[i];
}

static cudaError_t launch_untile(int bpp, const void* shards, size_t stride, int count, int only_rank, int width, int height, int tile, void* dst,
                                 cudaStream_t stream) {
    dim3 block(32, 8), grid((width + 31) / 32, (height + 7) / 8);
    const unsigned char* s = (const unsigned char*)shards;
    unsigned char* d = (unsigned char*)dst;
    if (bpp == 32) untile_kernel<32><<<grid, block, 0, stream>>>(s, stride, count, only_rank, width, height, tile, d);
    else if (bpp == 12) untile_kernel<12><<<grid, block, 0, stream>>>(s, stride, count, only_rank, width, height, tile, d);
    else if (bpp == 48) untile_kernel<48><<<grid, block, 0, stream>>>(s, stride, count, only_rank, width, height, tile, d);
    else untile_kernel<3><<<grid, block, 0, stream>>>(s, stride, count, only_rank, width, height, tile, d);
    return cudaGetLastError();
}

// The one way to the staging buffers for a writer on ctx->stream: out_lin / out_rgb8 of `pixels` slots and frame_scratch
// of `scratch_bytes` (full-frame copies of compact data, gathered sums), grown on demand.  The writer is ordered after
// the copy of every outstanding hand-out (rt_download_begin / rt_untile_begin), which reads these buffers until its
// rt_frame_end: a readback issued meanwhile does not change the frame the hand-out returns.
static int stage_buffers(DevCtx* ctx, size_t pixels, size_t scratch_bytes) {
    const bool grow_out = pixels > ctx->out_pixels, grow_scratch = scratch_bytes > ctx->frame_scratch_cap;
    if ((grow_out || grow_scratch) && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);  // no free under a running copy
    if (grow_out) {
        if (ctx->out_lin) cudaFree(ctx->out_lin);
        if (ctx->out_rgb8) cudaFree(ctx->out_rgb8);
        ctx->out_lin = nullptr;
        ctx->out_rgb8 = nullptr;
        ctx->out_pixels = 0;
        if (cudaMalloc(&ctx->out_lin, pixels * 3 * sizeof(float)) != cudaSuccess || cudaMalloc(&ctx->out_rgb8, pixels * 3) != cudaSuccess)
            return fail(ctx, RT_ERR_NOMEM, "rt_download: cannot allocate the output buffers");
        ctx->out_pixels = pixels;
    }
    if (grow_scratch) {
        if (ctx->frame_scratch) cudaFree(ctx->frame_scratch);
        ctx->frame_scratch = nullptr;
        ctx->frame_scratch_cap = 0;
        if (cudaMalloc(&ctx->frame_scratch, scratch_bytes) != cudaSuccess)
            return fail(ctx, RT_ERR_NOMEM, "cannot allocate %zu bytes of frame scratch", scratch_bytes);
        ctx->frame_scratch_cap = scratch_bytes;
    }
    for (const DevCtx::OutFrame& f : ctx->frames)
        if (f.active) CU(ctx, cudaStreamWaitEvent(ctx->stream, f.done, 0));
    return RT_OK;
}

// A plane of `bpp`-byte slots in layout L on the device -> the full row-major frame in host memory; a compact plane's
// tiles go to their places in a zeroed frame (black elsewhere).  Returns with ctx->stream synchronised.
static int plane_to_host(DevCtx* ctx, const void* plane, int bpp, const AccumLayout& L, void* host) {
    const size_t full = (size_t)L.width * L.height * bpp;
    if (L.compact) {
        int rc = stage_buffers(ctx, 0, full);
        if (rc != RT_OK) return rc;
        CU(ctx, cudaMemsetAsync(ctx->frame_scratch, 0, full, ctx->stream));
        CU(ctx, launch_untile(bpp, plane, 0, L.count, L.rank, L.width, L.height, L.tile, ctx->frame_scratch, ctx->stream));
        plane = ctx->frame_scratch;
    }
    CU(ctx, cudaMemcpyAsync(host, plane, full, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

static int dev_wait(DevCtx* ctx);

// Checkpoint / resume of a progressive render (SURVEY 8f rank 3): the frame so far IS the
// accumulation buffer (integer sums), so a raw copy of it plus the index of the next sample is a
// complete checkpoint, and a resumed render is bit-identical to an uninterrupted one.  Always the
// FULL row-major frame on the host side: a compact buffer is scattered into a zeroed frame first.
static int dev_accum_download(DevCtx* ctx, uint64_t* host, size_t bytes) {
    if (!ctx || !host) return RT_ERR_INVALID;
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "rt_accum_download: nothing rendered or bound yet");
    const size_t full = (size_t)ctx->acc.width * ctx->acc.height * 32;
    if (bytes < full) return fail(ctx, RT_ERR_INVALID, "rt_accum_download: need %zu bytes, got %zu", full, bytes);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    return plane_to_host(ctx, ctx->accum, 32, ctx->acc, host);
}

static int dev_accum_upload(DevCtx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height) {
    if (!ctx || !host) return RT_ERR_INVALID;
    if (width <= 0 || height <= 0 || (long long)width * height >= (1ll << 31)) return fail(ctx, RT_ERR_INVALID, "rt_accum_upload: bad frame size %dx%d", width, height);
    const size_t need = (size_t)width * height * 4 * sizeof(unsigned long long);
    if (bytes != need) return fail(ctx, RT_ERR_INVALID, "rt_accum_upload: a %dx%d frame is %zu bytes, got %zu", width, height, need, bytes);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    AccumLayout L;
    L.width = width;
    L.height = height;
    rc = ensure_accum(ctx, L);
    if (rc != RT_OK) return rc;
    // on the context's stream (cudaMemcpy from pageable memory returns once the data is STAGED; the DMA itself is
    // ordered only against the legacy stream, and ctx->stream is non-blocking: a render enqueued right after could
    // start before the sums have landed)
    CU(ctx, cudaMemcpyAsync(ctx->accum, host, need, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->moments_valid = false;  // until rt_moments_upload restores the moments of the same samples
    ctx->sums_uploaded = true;
    return RT_OK;
}

// Finish what an RT_FLAG_ASYNC render left pending: wait for the stream it ran on, read the device time and
// (STATS) the counters.  Everything that touches the frame or the scene calls this first.
static int dev_wait_lanes(DevCtx* ctx, float* ms_per_pass) {
    float ms_max = 0.0f;
    bool had = false;
    for (int k = 0; k < 2; k++) {
        if (!ctx->lane_busy[k]) continue;
        ctx->lane_busy[k] = false;
        had = true;
        CU(ctx, cudaEventSynchronize(ctx->lane_end[k]));
        float ms = 0.0f;
        CU(ctx, cudaEventElapsedTime(&ms, ctx->ov_begin, ctx->lane_end[k]));
        ms_max = std::max(ms_max, ms);
    }
    *ms_per_pass = had && ctx->ov_passes > 0 ? ms_max / (float)ctx->ov_passes : -1.0f;
    ctx->ov_passes = 0;
    return RT_OK;
}

static int dev_wait(DevCtx* ctx) {
    CU(ctx, cudaSetDevice(ctx->device));
    float ov_ms = -1.0f;
    int rcl = dev_wait_lanes(ctx, &ov_ms);  // overlapped passes (RT_FLAG_OVERLAP) first: they follow the pending plain pass
    if (rcl != RT_OK) return rcl;
    if (!ctx->pending_async) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (ov_ms >= 0.0f) ctx->stats.render_ms = ov_ms;
        return RT_OK;
    }
    ctx->pending_async = false;
    CU(ctx, cudaEventSynchronize(ctx->ev1));
    if (ctx->pending_stream != ctx->stream) CU(ctx, cudaStreamSynchronize(ctx->pending_stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    CU(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->stats.render_ms = ms;
    if (ov_ms >= 0.0f) ctx->stats.render_ms = ov_ms;
    if (ctx->pending_stats) {
        Stats h;
        CU(ctx, cudaMemcpyAsync(&h, ctx->dstats, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaMemcpyAsync(ctx->stats.trav_hist, ctx->dstats + 1, sizeof ctx->stats.trav_hist, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->stats.rays = h.rays;
        ctx->stats.node_visits = h.node_visits;
        ctx->stats.box_tests = h.box_tests;
        ctx->stats.sphere_tests = h.sphere_tests;
        ctx->stats.quad_tests = h.quad_tests;
        ctx->stats.triangle_tests = h.tri_tests;
        ctx->stats.medium_queries = h.medium_queries;
        ctx->stats.boundary_tests = h.boundary_tests;
        ctx->stats.fp64_sphere_tests = h.fp64_sphere;
        ctx->stats.empty_node_steps = h.empty_steps;
        ctx->stats.nonfinite_samples = h.nonfinite;
        ctx->stats.desc_iters = h.desc_iters;
        ctx->stats.desc_lanes = h.desc_lanes;
        ctx->stats.desc_trav_lanes = h.desc_trav_lanes;
        ctx->stats.leaf_iters = h.leaf_iters;
        ctx->stats.leaf_lanes = h.leaf_lanes;
        ctx->stats.shade_iters = h.shade_iters;
        ctx->stats.shade_lanes = h.shade_lanes;
    }
    return RT_OK;
}

// Orders `stream` (NULL: the context's own) after every render the context still has in flight -- the pending
// asynchronous pass and the RT_FLAG_OVERLAP passes on the lane streams.  No host wait.
static int dev_join(DevCtx* ctx, cudaStream_t stream) {
    if (!ctx) return RT_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!stream) stream = ctx->stream;
    for (int k = 0; k < 2; k++)
        if (ctx->lane_busy[k]) CU(ctx, cudaStreamWaitEvent(stream, ctx->lane_end[k], 0));
    if (ctx->pending_async && ctx->pending_stream != stream) CU(ctx, cudaStreamWaitEvent(stream, ctx->ev1, 0));
    return RT_OK;
}

static int dev_sync(DevCtx* ctx) {
    if (!ctx) return RT_ERR_INVALID;
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    CU(ctx, cudaDeviceSynchronize());
    return RT_OK;
}

// dynamic shared memory of a wide instance: the traversal stacks, [entry][thread]
static size_t v2_smem(const DevCtx* ctx, int width) { return width <= 2 ? 0 : (size_t)std::max(ctx->wide_depth, 1) * RT_V2_THREADS * sizeof(uint2); }

// the persistent grid of the instance: SMs x the blocks per SM it runs with
static int v2_grid(DevCtx* ctx, const V2Instance* e, int* grid) {
    if (!e) return fail(ctx, RT_ERR_UNSUPPORTED, "no compiled instance of render_kernel_v2 for this pass");
    const size_t smem = v2_smem(ctx, e->width);
    if (smem) {
        // carve out what RT_MIN_BLOCKS blocks need (plus the 1 KB the system reserves per block), the rest stays L1
        const int pct = (int)std::min<size_t>(100, (100 * RT_WIDE_MIN_BLOCKS * (smem + 1024) + 233471) / 233472);
        CU(ctx, cudaFuncSetAttribute((const void*)e->kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
    int bps = 0;
    CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, (const void*)e->kernel, RT_V2_THREADS, smem));
    *grid = ctx->sm_count * (bps > 0 ? bps : 1);
    return RT_OK;
}

static int launch_v2(DevCtx* ctx, const V2Instance& e, int grid, const RenderArgs& A, unsigned long long* accum,
                     unsigned long long* counters, cudaStream_t stream) {
    e.kernel<<<grid, RT_V2_THREADS, v2_smem(ctx, e.width), stream>>>(ctx->scene, A, accum, counters, ctx->dstats);
    CU(ctx, cudaGetLastError());
    return RT_OK;
}

// the checks of rt_render_params that rt_render and rt_render_views share; `entry` names the entry point in the messages
static int check_render_params(DevCtx* ctx, const rt_render_params* p, const char* entry) {
    if (!p || p->struct_size != sizeof(rt_render_params)) return fail(ctx, RT_ERR_INVALID, "%s: bad params struct", entry);
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "%s: no scene uploaded", entry);
    if (p->width <= 0 || p->height <= 0 || p->samples_per_pixel <= 0 || p->max_depth < 0 || p->spp_begin < 0)
        return fail(ctx, RT_ERR_INVALID, "%s: width/height/samples must be positive", entry);
    // a sample is clamped to 2^20 (kSampleClamp) and stored in 2^-28 units: 2^16 saturated samples fill a 64-bit sum
    if ((long long)p->spp_begin + p->samples_per_pixel > 65536)
        return fail(ctx, RT_ERR_UNSUPPORTED, "%s: samples %d + %d exceed 65536 per pixel, the capacity of the 64-bit fixed-point sums",
                    entry, p->spp_begin, p->samples_per_pixel);
    if (p->tile_size > 0 && p->tile_size % 8 != 0) return fail(ctx, RT_ERR_INVALID, "%s: tile_size must be a multiple of 8", entry);
    return RT_OK;
}

static int tile_size_of(const rt_render_params* p) { return p->tile_size > 0 ? p->tile_size : 16; }

// The shard mode a render of `count` shards runs: a single shard renders all tiles; RT_SHARD_AUTO shards tiles when every
// shard gets 256 or more of them, samples otherwise (sharding.py plans the same).  Any other mode is returned as given.
static int shard_mode_of(int width, int height, int tile, int count, int mode) {
    if (count == 1) return RT_SHARD_TILES;
    if (mode != RT_SHARD_AUTO) return mode;
    const long long n_tiles = (long long)((width + tile - 1) / tile) * ((height + tile - 1) / tile);
    return n_tiles / count >= 256 ? RT_SHARD_TILES : RT_SHARD_SAMPLES;
}

// The geometry of a pass: the tiles of the frame, the tiles or samples of shard `rank` of `count` (mode RT_SHARD_TILES or
// RT_SHARD_SAMPLES), and the (pixel block, sample segment) work items for a grid of `grid` blocks.  A batch of n_views
// frames (rt_render_views) is one shard whose local tiles are views x tiles, view-major.
static void plan_pass(RenderArgs& A, const rt_render_params* p, int mode, int rank, int count, int n_views, int grid) {
    std::memset(&A, 0, sizeof A);
    A.width = p->width;
    A.height = p->height;
    A.max_depth = p->max_depth;
    A.spp_begin = p->spp_begin;
    A.tile_size = tile_size_of(p);
    A.tiles_x = (p->width + A.tile_size - 1) / A.tile_size;
    A.tiles_y = (p->height + A.tile_size - 1) / A.tile_size;
    A.blocks_per_tile_x = A.tile_size / 8;
    A.blocks_per_tile_y = A.tile_size / 4;
    const int n_tiles = n_views * A.tiles_x * A.tiles_y;
    if (mode == RT_SHARD_TILES) {
        A.tile_stride = count;
        A.tile_offset = rank;
        A.n_local_tiles = (n_tiles - rank + count - 1) / count;
        A.sample_stride = 1;
        A.sample_offset = 0;
        A.n_local_samples = p->samples_per_pixel;
    } else {
        A.tile_stride = 1;
        A.tile_offset = 0;
        A.n_local_tiles = n_tiles;
        A.sample_stride = count;
        A.sample_offset = rank;
        A.n_local_samples = (p->samples_per_pixel - rank + count - 1) / count;  // 0 for a shard past the last sample
    }
    // segment length: enough work items to keep every resident warp busy ~64 times over,
    // but never shorter than 1 sample (fixed-point sums make the split result-neutral)
    const unsigned long long pixel_blocks = (unsigned long long)A.n_local_tiles * A.blocks_per_tile_x * A.blocks_per_tile_y;
    const unsigned long long resident_warps = (unsigned long long)grid * (RT_V2_THREADS / 32);
    int n_seg = 1;
    if (A.n_local_samples > 0 && pixel_blocks > 0) {
        // >= 64 items per resident warp: the end-of-kernel tail is one item long
        unsigned long long want = (resident_warps * 64 + pixel_blocks - 1) / pixel_blocks;
        if (want < 1) want = 1;
        if (want > (unsigned long long)A.n_local_samples) want = A.n_local_samples;
        n_seg = (int)want;
    }
    A.seg_len = A.n_local_samples > 0 ? (A.n_local_samples + n_seg - 1) / n_seg : 1;
    A.n_segments = A.n_local_samples > 0 ? (A.n_local_samples + A.seg_len - 1) / A.seg_len : 0;
    A.n_items = pixel_blocks * (unsigned long long)A.n_segments;
}

// The tail of a pass on `stream`, after the caller has queued its clears: reset the work counter, launch between ev0 and
// ev1 (nothing to launch for a shard without samples), account the pass and leave it pending, or wait for it
static int enqueue_pass(DevCtx* ctx, const V2Instance& e, int grid, const RenderArgs& A, unsigned long long* accum,
                        cudaStream_t stream, uint64_t samples, bool stats, bool async) {
    CU(ctx, cudaMemsetAsync(ctx->counters, 0, 4 * sizeof(unsigned long long), stream));
    CU(ctx, cudaEventRecord(ctx->ev0, stream));
    ctx->stats.kernel_launches = 0;
    if (A.n_items > 0) {
        int rc = launch_v2(ctx, e, grid, A, accum, ctx->counters, stream);
        if (rc != RT_OK) return rc;
        ctx->stats.kernel_launches = 1;
    }
    ctx->stats.blocks = grid;
    ctx->stats.samples = samples;
    CU(ctx, cudaEventRecord(ctx->ev1, stream));
    ctx->pending_async = true;
    ctx->pending_stats = stats;
    ctx->pending_stream = stream;
    if (async) return RT_OK;
    return dev_wait(ctx);
}

static int dev_render(DevCtx* ctx, const rt_render_params* p) {
    if (!ctx) return RT_ERR_INVALID;
    int rc = check_render_params(ctx, p, "rt_render");
    if (rc != RT_OK) return rc;
    if ((long long)p->width * p->height >= (1ll << 31)) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render: frame too large");
    const int count = p->shard_count <= 1 ? 1 : p->shard_count;
    const int rank = count == 1 ? 0 : p->shard_rank;
    if (rank < 0 || rank >= count) return fail(ctx, RT_ERR_INVALID, "rt_render: shard_rank %d outside [0,%d)", rank, count);
    const bool moments = (p->flags & RT_FLAG_MOMENTS) != 0;
    if (moments && (p->flags & RT_FLAG_STATS)) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render: RT_FLAG_MOMENTS has no RT_FLAG_STATS instance");
    if (moments && (p->flags & RT_FLAG_ACCUMULATE) && !ctx->moments_valid)
        return fail(ctx, RT_ERR_STATE, "rt_render: RT_FLAG_MOMENTS | RT_FLAG_ACCUMULATE onto a frame whose sums have no moments "
                                       "(start it with a non-accumulating moments pass, or restore both with rt_accum_upload + rt_moments_upload)");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t stream = p->stream ? (cudaStream_t)p->stream : ctx->stream;
    // RT_FLAG_OVERLAP: this pass goes to one of the two lane streams with its own work counter and waits for nothing on
    // the host; it needs the frame the passes before it render into, unchanged
    // (the camera of this frame size must be set up already: the first pass onto a restored checkpoint is a plain one)
    const bool overlap = (p->flags & RT_FLAG_OVERLAP) && (p->flags & RT_FLAG_ASYNC) && (p->flags & RT_FLAG_ACCUMULATE) &&
                         !(p->flags & RT_FLAG_STATS) && ctx->accum != nullptr &&
                         ctx->cam_w == p->width && ctx->cam_h == p->height;
    // a pending asynchronous render (possibly on another stream) shares the work counter, the guard flags and the
    // stats block with this one: finish it first
    rc = overlap ? RT_OK : dev_wait(ctx);
    if (rc != RT_OK) return rc;
    if (ctx->cam_w != p->width || ctx->cam_h != p->height) setup_camera(ctx, p->width, p->height);

    const int mode = shard_mode_of(p->width, p->height, tile_size_of(p), count, p->shard_mode);
    if (mode != RT_SHARD_TILES && mode != RT_SHARD_SAMPLES) return fail(ctx, RT_ERR_INVALID, "rt_render: unknown shard_mode %d", p->shard_mode);
    AccumLayout L;
    L.width = p->width;
    L.height = p->height;
    if (p->flags & RT_FLAG_COMPACT_TILES) {
        if (mode != RT_SHARD_TILES) return fail(ctx, RT_ERR_INVALID, "rt_render: RT_FLAG_COMPACT_TILES needs tile sharding (shard_mode RT_SHARD_TILES)");
        L.compact = true;
        L.rank = rank;
        L.count = count;
        L.tile = tile_size_of(p);
    }
    if ((p->flags & RT_FLAG_ACCUMULATE) && ctx->accum && !(ctx->acc == L))
        return fail(ctx, RT_ERR_STATE, "rt_render: RT_FLAG_ACCUMULATE onto a buffer of another frame size or tile layout");
    rc = ensure_accum(ctx, L);
    if (rc != RT_OK) return rc;
    if (moments && !(p->flags & RT_FLAG_ACCUMULATE)) {
        rc = ensure_moments(ctx, L.slots());
        if (rc != RT_OK) return rc;
    }
    ctx->moments_valid = moments;  // an accumulating moments pass was checked above; any pass without the flag invalidates them
    ctx->sums_uploaded = false;
    const bool stats = (p->flags & RT_FLAG_STATS) != 0;
    const bool want_nee = (p->flags & RT_FLAG_NEE) != 0 && ctx->scene.n_nee_lights > 0;
    const bool want_shadow = (p->flags & RT_FLAG_SHADOWED_POINT_LIGHTS) != 0 && ctx->scene.n_lights > 0;
    // which instance of render_kernel_v2 runs: LITE = no triangles, no point lights, no defocus blur in this scene (see
    // hit_prim); the NEE instances count no STATS; the first per-scene instance that covers the scene's features, unless
    // RT_B200_GENERAL_INSTANCE=1 asks for a general one
    const V2Key req{stats && !(want_nee || want_shadow), ctx->scene_lite && !getenv("RT_B200_NO_LITE"), want_nee || want_shadow, moments,
                    false, ctx->scene.wide_width ? ctx->scene.wide_width : 2, getenv("RT_B200_GENERAL_INSTANCE") ? FEAT_ALL : ctx->scene_feat};
    const V2Instance* e = v2_select(req);
    int grid = 0;
    rc = v2_grid(ctx, e, &grid);
    if (rc != RT_OK) return rc;
    RenderArgs A;
    plan_pass(A, p, mode, rank, count, 1, grid);
    A.compact = L.compact;
    A.set_side(ctx->moments);  // after ensure_moments: the first moments pass allocates the buffer
    A.nee_emitters = want_nee;
    A.shadow_point_lights = want_shadow;
    A.k0 = (uint32_t)(p->seed & 0xffffffffu);
    A.k1 = (uint32_t)(p->seed >> 32);

    // samples this pass traces: the whole frame, or the pixels of the tiles this shard owns
    auto pass_samples = [&]() -> uint64_t {
        if (!(mode == RT_SHARD_TILES && count > 1)) return (uint64_t)A.n_local_samples * (uint64_t)p->width * p->height;
        uint64_t px = 0;
        for (int t = rank; t < A.tiles_x * A.tiles_y; t += count) {
            int tx = t % A.tiles_x, ty = t / A.tiles_x;
            int w = std::min(A.tile_size, p->width - tx * A.tile_size), h = std::min(A.tile_size, p->height - ty * A.tile_size);
            px += (uint64_t)w * h;
        }
        return px * (uint64_t)A.n_local_samples;
    };
    if (overlap) {
        const int k = ctx->lane_next;
        ctx->lane_next ^= 1;
        if (!ctx->lane_stream[k]) {
            CU(ctx, cudaStreamCreateWithFlags(&ctx->lane_stream[k], cudaStreamNonBlocking));
            CU(ctx, cudaEventCreateWithFlags(&ctx->lane_end[k], cudaEventDefault));
        }
        if (!ctx->ev_fork) {
            CU(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
            CU(ctx, cudaEventCreate(&ctx->ov_begin));
        }
        cudaStream_t ls = ctx->lane_stream[k];
        unsigned long long* cnt = ctx->counters + 4 * (1 + k);
        // after everything `stream` holds now (the clearing pass, a restored checkpoint, ...); the previous pass of this
        // lane precedes this one in stream order, the pass on the other lane runs beside it
        CU(ctx, cudaEventRecord(ctx->ev_fork, stream));
        CU(ctx, cudaStreamWaitEvent(ls, ctx->ev_fork, 0));
        if (!ctx->lane_busy[0] && !ctx->lane_busy[1]) {
            CU(ctx, cudaEventRecord(ctx->ov_begin, ls));
            ctx->ov_passes = 0;
        }
        CU(ctx, cudaMemsetAsync(cnt, 0, 4 * sizeof(unsigned long long), ls));
        if (A.n_items > 0) {
            rc = launch_v2(ctx, *e, grid, A, ctx->accum, cnt, ls);
            if (rc != RT_OK) return rc;
        }
        CU(ctx, cudaEventRecord(ctx->lane_end[k], ls));
        ctx->lane_busy[k] = true;
        ctx->ov_passes++;
        ctx->stats.kernel_launches = A.n_items > 0 ? 1 : 0;
        ctx->stats.blocks = grid;
        ctx->stats.samples = pass_samples();
        return RT_OK;
    }
    if (!(p->flags & RT_FLAG_ACCUMULATE)) CU(ctx, cudaMemsetAsync(ctx->accum, 0, L.slots() * 32, stream));
    if (moments && !(p->flags & RT_FLAG_ACCUMULATE)) CU(ctx, cudaMemsetAsync(ctx->moments, 0, L.slots() * 48, stream));
    if (stats) CU(ctx, cudaMemsetAsync(ctx->dstats, 0, sizeof(Stats) + kTravHistBins * sizeof(unsigned long long), stream));
    return enqueue_pass(ctx, *e, grid, A, ctx->accum, stream, pass_samples(), stats, (p->flags & RT_FLAG_ASYNC) != 0);
}

// ---- multi-view batches (rt_render_views) ---------------------------------------------------------------------------
// n_views cameras of the uploaded scene in one launch of a VIEWS instance, into the views frame of the context.  View v
// runs the arithmetic of a single render with cameras[v] (camera_block, camera_ray) under the key of its seed, so it is
// bit-identical to that render: a sample is a pure function of (scene, camera, pixel, sample index, depth, key), and the
// sums are order-independent integers.
static int dev_render_views(DevCtx* ctx, const rt_render_params* p, const rt_camera* cameras, const uint64_t* seeds, int32_t n_views) {
    if (!ctx) return RT_ERR_INVALID;
    int rc = check_render_params(ctx, p, "rt_render_views");
    if (rc != RT_OK) return rc;
    if (n_views < 1 || !cameras) return fail(ctx, RT_ERR_INVALID, "rt_render_views: needs n_views >= 1 cameras (got %d%s)", n_views, cameras ? "" : ", NULL");
    const uint32_t unsupported = RT_FLAG_STATS | RT_FLAG_MOMENTS | RT_FLAG_COMPACT_TILES | RT_FLAG_OVERLAP;
    if ((p->flags & unsupported) || p->shard_count > 1)
        return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render_views: RT_FLAG_STATS, RT_FLAG_MOMENTS, RT_FLAG_COMPACT_TILES, RT_FLAG_OVERLAP and shards are not "
                                             "supported for multi-view batches (flags 0x%x, shard_count %d)", p->flags & unsupported, p->shard_count);
    if ((long long)n_views * p->width * p->height >= (1ll << 31))
        return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render_views: %d views of %dx%d are 2^31 slots or more", n_views, p->width, p->height);
    bool defocus = false;
    for (int v = 0; v < n_views; v++) {
        if (std::memcmp(cameras[v].background, ctx->camera.background, sizeof ctx->camera.background) != 0)
            return fail(ctx, RT_ERR_INVALID, "rt_render_views: the background of camera %d differs from the uploaded camera's (the scene keeps one background)", v);
        defocus = defocus || cameras[v].defocus_angle > 0;
    }
    // the views, their seeds and the frame shape: what an accumulating pass must continue
    uint64_t key = 0x5eed5eed00000000ull ^ (uint64_t)n_views;
    const int32_t shape[3] = {n_views, p->width, p->height};
    key = hash_bytes(key, shape, sizeof shape);
    key = hash_bytes(key, cameras, (size_t)n_views * sizeof(rt_camera));
    std::vector<ViewRecord> table((size_t)n_views);
    for (int v = 0; v < n_views; v++) {
        const uint64_t seed = seeds ? seeds[v] : p->seed;
        key = hash_bytes(key, &seed, sizeof seed);
        ViewRecord& R = table[v];
        std::memset(&R, 0, sizeof R);
        put_camera(R, camera_block(cameras[v], p->width, p->height));
        R.k0 = (uint32_t)(seed & 0xffffffffu);
        R.k1 = (uint32_t)(seed >> 32);
    }
    const bool accumulate = (p->flags & RT_FLAG_ACCUMULATE) != 0;
    if (accumulate && !(ctx->views_n > 0 && ctx->views_n == n_views && ctx->views_w == p->width && ctx->views_h == p->height && ctx->views_key == key))
        return fail(ctx, RT_ERR_STATE, "rt_render_views: RT_FLAG_ACCUMULATE onto a views frame of other views, size, cameras or seeds%s",
                    ctx->views_n > 0 ? "" : " (no views render yet)");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t stream = p->stream ? (cudaStream_t)p->stream : ctx->stream;
    // a pending asynchronous render shares the work counter and the events with this one; it may also still read the table
    rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    const size_t slots = (size_t)n_views * p->width * p->height;
    if (!ctx->views_accum || slots * 32 > ctx->views_cap) {
        if (ctx->views_accum) cudaFree(ctx->views_accum);
        ctx->views_accum = nullptr;
        ctx->views_cap = 0;
        ctx->views_n = 0;
        if (cudaMalloc(&ctx->views_accum, slots * 32) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "rt_render_views: cannot allocate %zu bytes for the views frame", slots * 32);
        ctx->views_cap = slots * 32;
    }
    if ((size_t)n_views * sizeof(ViewRecord) > ctx->view_table_cap) {
        if (ctx->view_table) cudaFree(ctx->view_table);
        ctx->view_table = nullptr;
        ctx->view_table_cap = 0;
        if (cudaMalloc(&ctx->view_table, (size_t)n_views * sizeof(ViewRecord)) != cudaSuccess)
            return fail(ctx, RT_ERR_NOMEM, "rt_render_views: cannot allocate the table of %d views", n_views);
        ctx->view_table_cap = (size_t)n_views * sizeof(ViewRecord);
    }
    // the single-frame path's background, whether or not rt_render has set up the camera since the upload
    put_background(ctx->scene, ctx->camera);

    const bool want_nee = (p->flags & RT_FLAG_NEE) != 0 && ctx->scene.n_nee_lights > 0;
    const bool want_shadow = (p->flags & RT_FLAG_SHADOWED_POINT_LIGHTS) != 0 && ctx->scene.n_lights > 0;
    // LITE only when no view needs the defocus code the LITE instance leaves out
    const V2Key req{false, ctx->geom_lite && !defocus && !getenv("RT_B200_NO_LITE"), want_nee || want_shadow, false, true, 2, FEAT_ALL};
    const V2Instance* e = v2_select(req);
    int grid = 0;
    rc = v2_grid(ctx, e, &grid);
    if (rc != RT_OK) return rc;
    RenderArgs A;
    plan_pass(A, p, RT_SHARD_TILES, 0, 1, n_views, grid);
    A.set_side(ctx->view_table);
    A.nee_emitters = want_nee;
    A.shadow_point_lights = want_shadow;

    CU(ctx, cudaMemcpyAsync(ctx->view_table, table.data(), table.size() * sizeof(ViewRecord), cudaMemcpyHostToDevice, stream));
    if (!accumulate) CU(ctx, cudaMemsetAsync(ctx->views_accum, 0, slots * 32, stream));
    ctx->views_n = n_views;
    ctx->views_w = p->width;
    ctx->views_h = p->height;
    ctx->views_key = key;
    // `table` may go with an asynchronous pass still queued: a copy from pageable memory has been staged when it returns
    return enqueue_pass(ctx, *e, grid, A, ctx->views_accum, stream, (uint64_t)slots * (uint64_t)p->samples_per_pixel, false,
                        (p->flags & RT_FLAG_ASYNC) != 0);
}

// resolve_kernel over `n` slots of sums (an accumulation buffer, a range of views, a gathered frame) into DEVICE buffers
static int dev_resolve_into(DevCtx* ctx, const unsigned long long* sums, size_t n, int32_t total_spp, float* dev_lin, unsigned char* dev_rgb8) {
    if (n == 0 || (!dev_lin && !dev_rgb8)) return RT_OK;
    const double inv = 1.0 / ((double)kAccumScale * (double)total_spp);
    resolve_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(sums, (int)n, inv, dev_lin, dev_rgb8);
    CU(ctx, cudaGetLastError());
    return RT_OK;
}

// The sums of layout L resolved into out_lin / out_rgb8 and copied to the host planes that are not null
static int resolve_to_host(DevCtx* ctx, const unsigned long long* sums, const AccumLayout& L, int32_t total_spp, float* rgb_linear, uint8_t* rgb8) {
    const size_t n = L.slots();
    int rc = stage_buffers(ctx, n, 0);
    if (rc == RT_OK) rc = dev_resolve_into(ctx, sums, n, total_spp, rgb_linear ? ctx->out_lin : nullptr, rgb8 ? ctx->out_rgb8 : nullptr);
    if (rc == RT_OK && rgb_linear) rc = plane_to_host(ctx, ctx->out_lin, 12, L, rgb_linear);
    if (rc == RT_OK && rgb8) rc = plane_to_host(ctx, ctx->out_rgb8, 3, L, rgb8);
    return rc;
}

// The compact tiles of this shard resolved into caller-owned DEVICE buffers (for a gather over NCCL by the caller:
// one process per GPU).  capacity_pixels >= rt_shard_pixels(...) of the rendered layout.
static int dev_resolve_tiles(DevCtx* ctx, int32_t total_spp, float* dev_rgb_linear, uint8_t* dev_rgb8, size_t capacity_pixels) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "rt_resolve_tiles: nothing rendered yet");
    if (total_spp <= 0) return fail(ctx, RT_ERR_INVALID, "rt_resolve_tiles: total_spp must be positive");
    if (capacity_pixels < ctx->acc.slots()) return fail(ctx, RT_ERR_INVALID, "rt_resolve_tiles: the buffers hold %zu pixels, the frame has %zu", capacity_pixels, ctx->acc.slots());
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    rc = dev_resolve_into(ctx, ctx->accum, ctx->acc.slots(), total_spp, dev_rgb_linear, dev_rgb8);
    if (rc != RT_OK) return rc;
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// Compact buffers of `shard_count` shards, gathered on this context's device (shard r at dev_shards + r * stride),
// scattered into the full row-major frame and copied to the host.  bytes_per_pixel 3, 12 or 32.
static int dev_untile(DevCtx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count, int32_t width,
                      int32_t height, int32_t tile_size, void* host_out) {
    if (!ctx || !dev_shards || !host_out) return RT_ERR_INVALID;
    if (width <= 0 || height <= 0 || tile_size <= 0 || shard_count <= 0 || (bytes_per_pixel != 3 && bytes_per_pixel != 12 && bytes_per_pixel != 32))
        return fail(ctx, RT_ERR_INVALID, "rt_untile: bad arguments");
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t full = (size_t)width * height * bytes_per_pixel;
    int rc = stage_buffers(ctx, 0, full);
    if (rc != RT_OK) return rc;
    CU(ctx, launch_untile(bytes_per_pixel, dev_shards, shard_stride_bytes, shard_count, -1, width, height, tile_size, ctx->frame_scratch, ctx->stream));
    CU(ctx, cudaMemcpyAsync(host_out, ctx->frame_scratch, full, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// ---- asynchronous hand-out ---------------------------------------------------------------------------------------
// begin: the frame is produced on ctx->stream (after whatever render is pending there or on the caller's stream), its
// copy to pinned host memory is queued on ctx->copy_stream, the call returns.  end: waits for the OLDEST outstanding
// begin and hands out pointers into the pinned buffer (valid until two more begins).  Two frames may be outstanding.
static int frame_slot(DevCtx* ctx, size_t px, bool lin, bool rgb8, DevCtx::OutFrame** out) {
    if (ctx->frames_out >= 2) return fail(ctx, RT_ERR_STATE, "two frames are already outstanding: call rt_frame_end first");
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    if (!ctx->ev_ready) CU(ctx, cudaEventCreateWithFlags(&ctx->ev_ready, cudaEventDisableTiming));
    DevCtx::OutFrame& f = ctx->frames[ctx->frame_head];
    if (!f.done) CU(ctx, cudaEventCreateWithFlags(&f.done, cudaEventDisableTiming));
    const size_t need = (lin ? px * 12 : 0) + 256 + (rgb8 ? px * 3 : 0);
    if (need > f.cap) {
        if (f.pinned) cudaFreeHost(f.pinned);
        f.pinned = nullptr;
        f.cap = 0;
        if (cudaHostAlloc(&f.pinned, need, cudaHostAllocDefault) != cudaSuccess) return fail(ctx, RT_ERR_NOMEM, "cannot allocate %zu bytes of pinned host memory", need);
        f.cap = need;
    }
    f.has_lin = lin;
    f.has_rgb8 = rgb8;
    f.off_lin = 0;
    f.off_rgb8 = lin ? ((px * 12 + 255) & ~(size_t)255) : 0;
    *out = &f;
    return RT_OK;
}
static int frame_queue_copy(DevCtx* ctx, DevCtx::OutFrame* f, const void* dev_lin, const void* dev_rgb8, size_t px) {
    CU(ctx, cudaEventRecord(ctx->ev_ready, ctx->stream));
    CU(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_ready, 0));
    if (f->has_lin) CU(ctx, cudaMemcpyAsync(f->pinned + f->off_lin, dev_lin, px * 12, cudaMemcpyDeviceToHost, ctx->copy_stream));
    if (f->has_rgb8) CU(ctx, cudaMemcpyAsync(f->pinned + f->off_rgb8, dev_rgb8, px * 3, cudaMemcpyDeviceToHost, ctx->copy_stream));
    CU(ctx, cudaEventRecord(f->done, ctx->copy_stream));
    f->active = true;
    ctx->frame_head ^= 1;
    ctx->frames_out++;
    return RT_OK;
}

static int dev_download_begin(DevCtx* ctx, int32_t total_spp, int32_t want_linear, int32_t want_rgb8) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "rt_download_begin: nothing rendered yet");
    if (total_spp <= 0 || (!want_linear && !want_rgb8)) return fail(ctx, RT_ERR_INVALID, "rt_download_begin: bad arguments");
    if (ctx->acc.compact) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_download_begin: compact tile buffers go through rt_resolve_tiles / rt_untile_begin");
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t px = ctx->acc.slots();
    DevCtx::OutFrame* f = nullptr;
    // stream order, no host wait: the previous copy and the pending render (on its own stream), then the resolve
    int rc = frame_slot(ctx, px, want_linear != 0, want_rgb8 != 0, &f);
    if (rc == RT_OK) rc = stage_buffers(ctx, px, 0);
    if (rc == RT_OK) rc = dev_join(ctx, ctx->stream);
    if (rc == RT_OK) rc = dev_resolve_into(ctx, ctx->accum, px, total_spp, want_linear ? ctx->out_lin : nullptr, want_rgb8 ? ctx->out_rgb8 : nullptr);
    if (rc != RT_OK) return rc;
    return frame_queue_copy(ctx, f, ctx->out_lin, ctx->out_rgb8, px);
}

static int dev_untile_begin(DevCtx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count, int32_t width,
                            int32_t height, int32_t tile_size) {
    if (!ctx || !dev_shards) return RT_ERR_INVALID;
    if (width <= 0 || height <= 0 || tile_size <= 0 || shard_count <= 0 || (bytes_per_pixel != 3 && bytes_per_pixel != 12))
        return fail(ctx, RT_ERR_INVALID, "rt_untile_begin: bad arguments (bytes_per_pixel 3 or 12)");
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t px = (size_t)width * height;
    DevCtx::OutFrame* f = nullptr;
    int rc = frame_slot(ctx, px, bytes_per_pixel == 12, bytes_per_pixel == 3, &f);
    if (rc == RT_OK) rc = stage_buffers(ctx, 0, px * bytes_per_pixel);
    if (rc != RT_OK) return rc;
    CU(ctx, launch_untile(bytes_per_pixel, dev_shards, shard_stride_bytes, shard_count, -1, width, height, tile_size, ctx->frame_scratch, ctx->stream));
    return frame_queue_copy(ctx, f, ctx->frame_scratch, ctx->frame_scratch, px);
}

static int dev_frame_end(DevCtx* ctx, const float** rgb_linear, const uint8_t** rgb8) {
    if (!ctx) return RT_ERR_INVALID;
    if (ctx->frames_out <= 0) return fail(ctx, RT_ERR_STATE, "rt_frame_end: no frame is outstanding");
    CU(ctx, cudaSetDevice(ctx->device));
    DevCtx::OutFrame& f = ctx->frames[ctx->frames_out == 2 ? ctx->frame_head : (ctx->frame_head ^ 1)];
    CU(ctx, cudaEventSynchronize(f.done));
    f.active = false;
    ctx->frames_out--;
    if (rgb_linear) *rgb_linear = f.has_lin ? (const float*)(f.pinned + f.off_lin) : nullptr;
    if (rgb8) *rgb8 = f.has_rgb8 ? (const uint8_t*)(f.pinned + f.off_rgb8) : nullptr;
    return RT_OK;
}

static int dev_download(DevCtx* ctx, int32_t total_spp, float* rgb_linear, uint8_t* rgb8) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "rt_download: nothing rendered yet");
    if (total_spp <= 0) return fail(ctx, RT_ERR_INVALID, "rt_download: total_spp must be positive");
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    return resolve_to_host(ctx, ctx->accum, ctx->acc, total_spp, rgb_linear, rgb8);
}

// views [first, first + count) of the views frame, each resolved like rt_download's planes
static int dev_download_views(DevCtx* ctx, int32_t total_spp, int32_t first, int32_t count, float* rgb_linear, uint8_t* rgb8) {
    if (!ctx) return RT_ERR_INVALID;
    if (ctx->views_n <= 0) return fail(ctx, RT_ERR_STATE, "rt_download_views: no views rendered yet");
    if (total_spp <= 0) return fail(ctx, RT_ERR_INVALID, "rt_download_views: total_spp must be positive");
    if (first < 0 || count < 1 || (long long)first + count > ctx->views_n)
        return fail(ctx, RT_ERR_INVALID, "rt_download_views: views [%d, %d + %d) outside the frame's %d views", first, first, count, ctx->views_n);
    int rc = dev_wait(ctx);
    if (rc != RT_OK) return rc;
    if (!rgb_linear && !rgb8) return RT_OK;
    // consecutive views of one size are one full frame views_w x (views_h * count)
    return resolve_to_host(ctx, ctx->views_accum + (size_t)first * ctx->views_w * ctx->views_h * 4, AccumLayout{ctx->views_w, ctx->views_h * count},
                           total_spp, rgb_linear, rgb8);
}

// ---- second moments (RT_FLAG_MOMENTS) ------------------------------------------------------------------------------
static int moments_ready(DevCtx* ctx, const char* what) {
    if (!ctx->accum) return fail(ctx, RT_ERR_STATE, "%s: nothing rendered yet", what);
    if (!ctx->moments_valid) return fail(ctx, RT_ERR_STATE, "%s: the frame has no moments (render it with RT_FLAG_MOMENTS)", what);
    return dev_wait(ctx);
}

// variance_kernel over the slots of the frame into out_lin (the buffer of the linear radiance of rt_download)
static int dev_variance_into(DevCtx* ctx, int32_t total_spp) {
    const size_t n = ctx->acc.slots();
    int rc = stage_buffers(ctx, n, 0);
    if (rc != RT_OK) return rc;
    if (n) variance_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->accum, ctx->moments, (int)n, total_spp, ctx->out_lin);
    CU(ctx, cudaGetLastError());
    return RT_OK;
}

static int dev_download_variance(DevCtx* ctx, int32_t total_spp, float* variance) {
    if (!ctx || !variance) return RT_ERR_INVALID;
    if (total_spp < 2) return fail(ctx, RT_ERR_INVALID, "rt_download_variance: total_spp must be at least 2");
    int rc = moments_ready(ctx, "rt_download_variance");
    if (rc == RT_OK) rc = dev_variance_into(ctx, total_spp);
    if (rc != RT_OK) return rc;
    return plane_to_host(ctx, ctx->out_lin, 12, ctx->acc, variance);
}

// the 12 integer partials of noise_kernel over the slots of this device, and the frame pixels they cover
static int dev_noise_partials(DevCtx* ctx, int32_t total_spp, uint64_t* partials, uint64_t* pixels) {
    int rc = moments_ready(ctx, "rt_frame_noise");
    if (rc != RT_OK) return rc;
    if (!ctx->noise_sums) CU(ctx, cudaMalloc(&ctx->noise_sums, 12 * sizeof(unsigned long long)));
    CU(ctx, cudaMemsetAsync(ctx->noise_sums, 0, 12 * sizeof(unsigned long long), ctx->stream));
    const size_t n = ctx->acc.slots();
    if (n) noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->accum, ctx->moments, (int)n, total_spp, ctx->noise_sums);
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(partials, ctx->noise_sums, 12 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    *pixels = ctx->acc.pixels();
    return RT_OK;
}

// the partials -> (mean linear radiance, RMS standard error of the pixel mean), the one division of rt_frame_noise
static void noise_from_partials(const uint64_t* w, uint64_t pixels, int32_t total_spp, double* mean, double* rms) {
    unsigned __int128 s1 = 0, q = 0;
    for (int c = 0; c < 3; c++) {
        s1 += (unsigned __int128)w[2 * c] + ((unsigned __int128)w[2 * c + 1] << 32);
        q += (unsigned __int128)w[6 + 2 * c] + ((unsigned __int128)w[7 + 2 * c] << 32);
    }
    const double values = 3.0 * (double)pixels;
    *mean = pixels ? (double)s1 / ((double)kAccumScale * (double)total_spp * values) : 0.0;
    *rms = pixels ? std::sqrt(std::ldexp((double)q, -kNoiseFracBits) / values) : 0.0;
}

static int dev_moments_download(DevCtx* ctx, uint64_t* host, size_t bytes) {
    if (!ctx || !host) return RT_ERR_INVALID;
    const size_t full = (size_t)ctx->acc.width * ctx->acc.height * 48;
    if (ctx->accum && bytes != full) return fail(ctx, RT_ERR_INVALID, "rt_moments_download: a %dx%d frame is %zu bytes, got %zu", ctx->acc.width, ctx->acc.height, full, bytes);
    int rc = moments_ready(ctx, "rt_moments_download");
    if (rc != RT_OK) return rc;
    return plane_to_host(ctx, ctx->moments, 48, ctx->acc, host);
}

// the moments of the sums rt_accum_upload restored just before (same full frame)
static int dev_moments_upload(DevCtx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height) {
    if (!ctx || !host) return RT_ERR_INVALID;
    if (width <= 0 || height <= 0 || (long long)width * height >= (1ll << 31)) return fail(ctx, RT_ERR_INVALID, "rt_moments_upload: bad frame size %dx%d", width, height);
    const size_t need = (size_t)width * height * 48;
    if (bytes != need) return fail(ctx, RT_ERR_INVALID, "rt_moments_upload: a %dx%d frame is %zu bytes, got %zu", width, height, need, bytes);
    if (!ctx->sums_uploaded || ctx->acc.compact || ctx->acc.width != width || ctx->acc.height != height)
        return fail(ctx, RT_ERR_STATE, "rt_moments_upload: follows rt_accum_upload of the same %dx%d frame", width, height);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = dev_wait(ctx);
    if (rc == RT_OK) rc = ensure_moments(ctx, (size_t)width * height);
    if (rc != RT_OK) return rc;
    CU(ctx, cudaMemcpyAsync(ctx->moments, host, need, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->moments_valid = true;
    return RT_OK;
}

static int dev_render_aov(DevCtx* ctx, int32_t width, int32_t height, int32_t* prim_id, float* t, float* normal, float* point,
                             float* uv) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_render_aov: no scene uploaded");
    if (width <= 0 || height <= 0) return fail(ctx, RT_ERR_INVALID, "rt_render_aov: bad frame size");
    CU(ctx, cudaSetDevice(ctx->device));
    if (ctx->cam_w != width || ctx->cam_h != height) setup_camera(ctx, width, height);
    const size_t n = (size_t)width * height;
    int* d_id = nullptr;
    float *d_t = nullptr, *d_n = nullptr, *d_p = nullptr, *d_uv = nullptr;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void** p, size_t bytes, const void* want) {
        if (want && e == cudaSuccess) e = cudaMalloc(p, bytes);
    };
    alloc((void**)&d_id, n * 4, prim_id);
    alloc((void**)&d_t, n * 4, t);
    alloc((void**)&d_n, n * 12, normal);
    alloc((void**)&d_p, n * 12, point);
    alloc((void**)&d_uv, n * 8, uv);
    if (e == cudaSuccess) {
        dim3 block(8, 8), grid((width + 7) / 8, (height + 7) / 8);
        aov_kernel<<<grid, block, 0, ctx->stream>>>(ctx->scene, ctx->camera_d, width, height, d_id, d_t, d_n, d_p, d_uv);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    auto fetch = [&](void* dst, const void* src, size_t bytes) {
        if (dst && e == cudaSuccess) e = cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
    };
    fetch(prim_id, d_id, n * 4);
    fetch(t, d_t, n * 4);
    fetch(normal, d_n, n * 12);
    fetch(point, d_p, n * 12);
    fetch(uv, d_uv, n * 8);
    cudaFree(d_id); cudaFree(d_t); cudaFree(d_n); cudaFree(d_p); cudaFree(d_uv);
    if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, "rt_render_aov: %s", cudaGetErrorString(e));
    return RT_OK;
}

static int dev_get_stats(DevCtx* ctx, rt_stats* out) {
    if (!ctx || !out) return RT_ERR_INVALID;
    *out = ctx->stats;
    return RT_OK;
}

extern "C" size_t rt_struct_size(int which) {
    static const size_t sizes[] = {sizeof(rt_scene_desc), sizeof(rt_render_params), sizeof(rt_stats), sizeof(rt_sphere), sizeof(rt_quad),
                                   sizeof(rt_triangle), sizeof(rt_medium), sizeof(rt_material), sizeof(rt_texture), sizeof(rt_image),
                                   sizeof(rt_perlin), sizeof(rt_point_light), sizeof(rt_camera), sizeof(rt_xform), sizeof(rt_prim_ref),
                                   sizeof(rt_mesh)};
    return (which >= 0 && which < (int)(sizeof(sizes) / sizeof(sizes[0]))) ? sizes[which] : 0;
}

static int dev_measure_fp32_peak(DevCtx* ctx, double* tflops) {
    if (!ctx || !tflops) return RT_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    float* d = nullptr;
    CU(ctx, cudaMalloc(&d, 16));
    const int iters = 1 << 16, threads = 1024, blocks = ctx->sm_count * 2;
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(ctx->ev0, ctx->stream);
        fma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(d, iters, 1.0000001f, 1e-7f);
        cudaEventRecord(ctx->ev1, ctx->stream);
        cudaError_t e = cudaEventSynchronize(ctx->ev1);
        if (e != cudaSuccess) { cudaFree(d); return fail(ctx, RT_ERR_CUDA, "rt_measure_fp32_peak: %s", cudaGetErrorString(e)); }
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        double flops = 2.0 * 8.0 * iters * (double)threads * blocks;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) * 1e-12);
    }
    cudaFree(d);
    *tflops = best;
    return RT_OK;
}

static int dev_measure_l1_peak(DevCtx* ctx, double* gbs) {
    if (!ctx || !gbs) return RT_ERR_INVALID;
    CU(ctx, cudaSetDevice(ctx->device));
    const int blocks = ctx->sm_count * 2, threads = 256, iters = 1 << 13;
    uint4* d = nullptr;
    const size_t bytes = (size_t)blocks * 2048 * sizeof(uint4);
    CU(ctx, cudaMalloc(&d, bytes + 64));
    cudaMemsetAsync(d, 1, bytes + 64, ctx->stream);
    cudaFuncSetAttribute(l1_peak_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 0);
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(ctx->ev0, ctx->stream);
        l1_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(d, iters, d + (bytes / sizeof(uint4)));
        cudaEventRecord(ctx->ev1, ctx->stream);
        cudaError_t e = cudaEventSynchronize(ctx->ev1);
        if (e != cudaSuccess) { cudaFree(d); return fail(ctx, RT_ERR_CUDA, "rt_measure_l1_peak: %s", cudaGetErrorString(e)); }
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        const double moved = 16.0 * 8.0 * iters * (double)threads * blocks;
        if (rep > 0) best = std::max(best, moved / (ms * 1e-3) * 1e-9);
    }
    cudaFree(d);
    *gbs = best;
    return RT_OK;
}

// ---- probes -----------------------------------------------------------------------
template <class Launch>
static int run_probe(DevCtx* ctx, const char* name, const std::vector<std::pair<const void*, size_t>>& inputs,
                     const std::vector<std::pair<void*, size_t>>& outputs, Launch launch) {
    CU(ctx, cudaSetDevice(ctx->device));
    std::vector<void*> din(inputs.size(), nullptr), dout(outputs.size(), nullptr);
    cudaError_t e = cudaSuccess;
    for (size_t i = 0; i < inputs.size() && e == cudaSuccess; i++) {
        e = cudaMalloc(&din[i], std::max<size_t>(inputs[i].second, 16));
        // stream-ordered with the probe kernel (a plain cudaMemcpy from pageable memory only guarantees staging:
        // the kernel on the non-blocking ctx->stream could read the buffer before the DMA lands)
        if (e == cudaSuccess && inputs[i].second) e = cudaMemcpyAsync(din[i], inputs[i].first, inputs[i].second, cudaMemcpyHostToDevice, ctx->stream);
    }
    for (size_t i = 0; i < outputs.size() && e == cudaSuccess; i++)
        if (outputs[i].first) e = cudaMalloc(&dout[i], std::max<size_t>(outputs[i].second, 16));
    if (e == cudaSuccess) {
        launch(din, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    for (size_t i = 0; i < outputs.size() && e == cudaSuccess; i++)
        if (outputs[i].first) e = cudaMemcpy(outputs[i].first, dout[i], outputs[i].second, cudaMemcpyDeviceToHost);
    for (void* p : din) cudaFree(p);
    for (void* p : dout) cudaFree(p);
    if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e));
    return RT_OK;
}

static int dev_probe_texture(DevCtx* ctx, int32_t texture, int32_t n, const float* uvp, float* rgb) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_probe_texture: no scene uploaded");
    if (n <= 0 || !uvp || !rgb) return fail(ctx, RT_ERR_INVALID, "rt_probe_texture: bad arguments");
    if (texture < 0 || texture >= ctx->n_textures) return fail(ctx, RT_ERR_INVALID, "rt_probe_texture: texture %d outside [0,%d)", texture, ctx->n_textures);
    return run_probe(ctx, "rt_probe_texture", {{uvp, (size_t)n * 20}}, {{rgb, (size_t)n * 12}},
                     [&](std::vector<void*>& in, std::vector<void*>& out) {
                         probe_texture_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene, texture, n, (const float*)in[0], (float*)out[0]);
                     });
}

static int dev_probe_scatter(DevCtx* ctx, int32_t material, int32_t n, const float* in_rec, const float* uniforms, float* out_rec) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_probe_scatter: no scene uploaded");
    if (n <= 0 || !in_rec || !uniforms || !out_rec) return fail(ctx, RT_ERR_INVALID, "rt_probe_scatter: bad arguments");
    if (material < 0 || material >= ctx->n_materials) return fail(ctx, RT_ERR_INVALID, "rt_probe_scatter: material %d outside [0,%d)", material, ctx->n_materials);
    return run_probe(ctx, "rt_probe_scatter", {{in_rec, (size_t)n * 64}, {uniforms, (size_t)n * 16}}, {{out_rec, (size_t)n * 64}},
                     [&](std::vector<void*>& in, std::vector<void*>& out) {
                         probe_scatter_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene, material, n, (const float*)in[0],
                                                                                         (const float*)in[1], (float*)out[0]);
                     });
}

static int dev_probe_hit(DevCtx* ctx, int32_t n, const float* rays, int32_t* prim_id, float* t, float* normal, float* uv) {
    if (!ctx) return RT_ERR_INVALID;
    if (!ctx->has_scene) return fail(ctx, RT_ERR_STATE, "rt_probe_hit: no scene uploaded");
    if (n <= 0 || !rays) return fail(ctx, RT_ERR_INVALID, "rt_probe_hit: bad arguments");
    int rc = run_probe(ctx, "rt_probe_hit", {{rays, (size_t)n * 36}},
                       {{prim_id, (size_t)n * 4}, {t, (size_t)n * 4}, {normal, (size_t)n * 12}, {uv, (size_t)n * 8}},
                       [&](std::vector<void*>& in, std::vector<void*>& out) {
                           probe_hit_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->scene, n, (const float*)in[0], (int*)out[0],
                                                                                       (float*)out[1], (float*)out[2], (float*)out[3]);
                       });
    return rc;
}

#include "rt_api.cuh"
