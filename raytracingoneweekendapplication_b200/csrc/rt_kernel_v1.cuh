// rt_kernel_v1.cuh -- the first megakernel (one lane = one pixel x a fixed share of samples, with
// path regeneration).  ncu measured 7.8 of 32 threads active per issued instruction
// (profiles/r1_v1_*); render_kernel_v2 replaced it.  Compiled only with -DRT_B200_ALT_KERNELS and
// selected with RT_B200_KERNEL=v1, for A/B measurements.  Included by rt_b200.cu after RenderArgs.
#pragma once

template <bool STATS>
__global__ void __launch_bounds__(256) render_kernel(const __grid_constant__ DevScene S, const __grid_constant__ RenderArgs A,
                                                     unsigned long long* __restrict__ accum,
                                                     unsigned long long* __restrict__ counters, Stats* __restrict__ gstats) {
    const unsigned lane = threadIdx.x & 31u;
    Stats st;
    if (STATS) memset(&st, 0, sizeof st);
    unsigned long long dropped = 0;

    while (true) {
        // one work item per warp: an 8x4 pixel block x one segment of samples
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(&counters[0], 1ull);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= A.n_items) break;

        const unsigned seg = (unsigned)(item % (unsigned long long)A.n_segments);
        unsigned long long blk = item / (unsigned long long)A.n_segments;
        const unsigned blocks_per_tile = (unsigned)(A.blocks_per_tile_x * A.blocks_per_tile_y);
        const unsigned local_tile = (unsigned)(blk / blocks_per_tile);
        const unsigned in_tile = (unsigned)(blk % blocks_per_tile);
        const unsigned tile = A.tile_offset + local_tile * A.tile_stride;
        const int tx = tile % A.tiles_x, ty = tile / A.tiles_x;
        const int bx = in_tile % A.blocks_per_tile_x, by = in_tile / A.blocks_per_tile_x;
        const int px = tx * A.tile_size + bx * 8 + (int)(lane & 7u);
        const int py = ty * A.tile_size + by * 4 + (int)(lane >> 3);
        const bool inside = px < A.width && py < A.height && (bx * 8 + (int)(lane & 7u)) < A.tile_size &&
                            (by * 4 + (int)(lane >> 3)) < A.tile_size;
        const uint32_t pixel = (uint32_t)(py * A.width + px);

        int s = (int)seg * A.seg_len;
        // ray_color(depth <= 0) is black before anything is traced (Camera.txt:205-206)
        const int s_end = (inside && A.max_depth > 0) ? min(s + A.seg_len, A.n_local_samples) : s;

        unsigned long long sum_r = 0, sum_g = 0, sum_b = 0;
        Rng rng;
        rng.pixel = pixel;
        rng.k0 = A.k0;
        rng.k1 = A.k1;
        rng.sample = 0;
        Ray ray;
        V3 L = v3(0, 0, 0), T = v3(1, 1, 1);
        uint32_t bounce = 0, origin_prim = PRIM_NONE;
        bool alive = false;

        while (true) {
            if (!alive) {
                if (s >= s_end) break;
                rng.sample = (uint32_t)(A.spp_begin + A.sample_offset + s * A.sample_stride);
                ray = camera_ray(S, px, py, rng);
                L = v3(0, 0, 0);
                T = v3(1, 1, 1);
                bounce = 0;
                origin_prim = PRIM_NONE;
                alive = true;
                if (STATS) st.samples++;
            }
            // ---- one bounce: Camera.txt:203-238 ------------------------------------
            Hit hit;
            traverse<STATS>(S, ray, 0.001f, __int_as_float(0x7f800000), origin_prim, hit, &st);
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
                    sf.p = fma3(hit.t, ray.d, ray.o);
                    sf.normal = v3(md.normal);
                    sf.front = true;
                    sf.u = sf.v = 0.0f;
                    sf.material = md.material;
                    sf.prim_id = -1;
                    origin_prim = PRIM_NONE;
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
                    if (bounce >= (uint32_t)A.max_depth) done = true;  // ray_color(depth <= 0) returns 0
                }
            }
            if (done) {
                const bool finite = isfinite(L.x) && isfinite(L.y) && isfinite(L.z);
                if (finite) {
                    sum_r += __float2ull_rn(fminf(fmaxf(L.x, 0.0f), kSampleClamp) * kAccumScale);
                    sum_g += __float2ull_rn(fminf(fmaxf(L.y, 0.0f), kSampleClamp) * kAccumScale);
                    sum_b += __float2ull_rn(fminf(fmaxf(L.z, 0.0f), kSampleClamp) * kAccumScale);
                } else {
                    dropped++;
                }
                alive = false;
                s++;
            }
        }
        if (inside) {
            unsigned long long* a = accum + 4ull * pixel;
            atomicAdd(a + 0, sum_r);
            atomicAdd(a + 1, sum_g);
            atomicAdd(a + 2, sum_b);
            if (dropped) { atomicAdd(a + 3, dropped); }
        }
        if (STATS) st.nonfinite += dropped;
        dropped = 0;
        __syncwarp();
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

