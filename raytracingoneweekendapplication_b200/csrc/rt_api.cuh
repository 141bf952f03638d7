// rt_api.cuh — the exported C ABI of include/rt_b200.h on top of the per-device layer of rt_b200.cu
// (included at its end).
//
// A context drives ONE OR SEVERAL GPUs of one box from one process (SURVEY 8b / 8e; replaces the reference's
// row bands over CPU threads, Camera.txt:59-61, 96-100):
//   * the scene is replicated: rt_upload_scene uploads (and, for big scenes, builds) and rt_refit_scene refits on
//     every device, in parallel host threads;
//   * rt_render cuts the frame into tile x tile tiles, tile t -> device t mod n (small frames: sample
//     s -> device s mod n), every device renders into a COMPACT buffer that holds only its own tiles
//     (1 / n of the frame), all devices run concurrently on their own streams;
//   * rt_download resolves every device's tiles on that device (sums -> RGB8 / float), gathers the resolved
//     tiles on device 0 over NVLink -- ncclSend / ncclRecv in one group when libnccl.so.2 can be loaded
//     (dlopen: the library has no link-time dependency on NCCL), cudaMemcpyPeerAsync otherwise -- scatters them
//     into the row-major frame there and copies it to the host.
// The image is bit-identical for any number of devices: a sample is a pure function of its Philox counter and
// the frame is a sum of integers.
#pragma once
#include <dlfcn.h>

#include <thread>

struct NcclApi {
    // the handful of NCCL entry points the gather uses, resolved at run time
    typedef struct ncclComm* comm_t;
    int (*CommInitAll)(comm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(comm_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*Send)(const void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    void* handle = nullptr;
    bool load() {
        if (handle) return true;
        handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!handle) return false;
        CommInitAll = (decltype(CommInitAll))dlsym(handle, "ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))dlsym(handle, "ncclCommDestroy");
        GroupStart = (decltype(GroupStart))dlsym(handle, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(handle, "ncclGroupEnd");
        Send = (decltype(Send))dlsym(handle, "ncclSend");
        Recv = (decltype(Recv))dlsym(handle, "ncclRecv");
        GetErrorString = (decltype(GetErrorString))dlsym(handle, "ncclGetErrorString");
        if (CommInitAll && CommDestroy && GroupStart && GroupEnd && Send && Recv) return true;
        dlclose(handle);
        handle = nullptr;
        return false;
    }
};
constexpr int kNcclUint8 = 1;  // ncclUint8 (nccl.h: ncclInt8 0, ncclUint8 1, ...)

struct rt_ctx {
    std::vector<DevCtx*> dev;
    std::string error;
    // multi-device state
    bool rendered = false;
    rt_render_params last{};      // the frame the devices hold (resolved shard mode and tile size)
    DeviceBuffer<unsigned char> gather;           // device 0: the shards' data side by side, shard d at d * gather_stride
    DeviceBuffer<unsigned long long> base_sums;  // device 0: a restored checkpoint (full frame), added to what the devices render
    int base_w = 0, base_h = 0;
    NcclApi nccl;
    std::vector<NcclApi::comm_t> comms;
    int gather_mode = 0;  // 0 peer copies, 1 NCCL send/recv
    uint32_t gathers = 0;
};

static int failx(rt_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->error = buf;
    return code;
}
// forwards a per-device status, keeping its message
static int fwd(rt_ctx* ctx, DevCtx* d, int rc) {
    if (rc != RT_OK && d) ctx->error = d->error;
    return rc;
}
#define CUX(ctx, call)                                                                                      \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) return failx(ctx, RT_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));     \
    } while (0)

extern "C" int rt_create(rt_ctx** out, const int* device_ids, int n_devices) {
    if (!out) return RT_ERR_INVALID;
    *out = nullptr;
    rt_ctx* ctx = new (std::nothrow) rt_ctx();
    if (!ctx) return RT_ERR_NOMEM;
    *out = ctx;  // returned even on failure so that rt_last_error works; the caller destroys it
    if (n_devices < 1 || n_devices > 64 || !device_ids) return failx(ctx, RT_ERR_INVALID, "rt_create: 1 to 64 devices (got %d)", n_devices);
    // RT_B200_ALLOW_DUPLICATE_DEVICES=1: a test hook -- the same GPU listed several times behaves like several GPUs
    // (own streams and buffers, gather by copies), so the multi-device path can be exercised on a one-GPU box
    const bool dup_ok = getenv("RT_B200_ALLOW_DUPLICATE_DEVICES") != nullptr;
    bool has_dup = false;
    for (int i = 0; i < n_devices; i++)
        for (int j = 0; j < i; j++)
            if (device_ids[i] == device_ids[j]) {
                if (!dup_ok) return failx(ctx, RT_ERR_INVALID, "rt_create: device %d listed twice", device_ids[i]);
                has_dup = true;
            }
    for (int i = 0; i < n_devices; i++) {
        DevCtx* d = nullptr;
        int rc = dev_create(&d, device_ids + i, 1);
        if (d) ctx->dev.push_back(d);
        if (rc != RT_OK) return fwd(ctx, d, rc);
    }
    if (n_devices > 1) {
        // device 0 reads the other devices' tiles: peer access where the hardware offers it (NVLink / NVSwitch)
        for (int i = 1; i < n_devices; i++) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, device_ids[0], device_ids[i]);
            if (can && device_ids[i] != device_ids[0]) {
                cudaSetDevice(device_ids[0]);
                cudaError_t e = cudaDeviceEnablePeerAccess(device_ids[i], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                cudaSetDevice(device_ids[i]);
                e = cudaDeviceEnablePeerAccess(device_ids[0], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            }
        }
        cudaGetLastError();
        const char* g = getenv("RT_B200_GATHER");  // nccl | p2p; default: NCCL when it loads
        const bool want_nccl = (!g || strcmp(g, "nccl") == 0) && !has_dup;  // NCCL refuses one GPU in two ranks
        if (want_nccl && ctx->nccl.load()) {
            ctx->comms.assign((size_t)n_devices, nullptr);
            if (ctx->nccl.CommInitAll(ctx->comms.data(), n_devices, device_ids) == 0) ctx->gather_mode = 1;
            else ctx->comms.clear();
        }
        if (g && strcmp(g, "nccl") == 0 && ctx->gather_mode != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_create: RT_B200_GATHER=nccl but libnccl.so.2 is not usable");
    }
    return RT_OK;
}

extern "C" void rt_destroy(rt_ctx* ctx) {
    if (!ctx) return;
    if (!ctx->dev.empty()) {
        cudaSetDevice(ctx->dev[0]->device);
        cudaDeviceSynchronize();
        ctx->gather.release();
        ctx->base_sums.release();
    }
    for (auto c : ctx->comms)
        if (c) ctx->nccl.CommDestroy(c);
    for (DevCtx* d : ctx->dev) dev_destroy(d);
    delete ctx;
}

extern "C" const char* rt_last_error(const rt_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }

extern "C" int rt_device_count(const rt_ctx* ctx) { return ctx ? (int)ctx->dev.size() : 0; }
extern "C" int rt_visible_devices(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

#define RT_NEED(ctx)                                        \
    if (!(ctx)) return RT_ERR_INVALID;                      \
    if ((ctx)->dev.empty()) return failx(ctx, RT_ERR_STATE, "the context was not created")

// An ABI-3 description ends where `meshes` begins: read no byte past its struct_size, take it as a scene without meshes
static const rt_scene_desc* widen_v3(const rt_scene_desc* sc, rt_scene_desc* v3) {
    if (!sc || sc->abi_version != 3 || sc->struct_size != offsetof(rt_scene_desc, meshes)) return sc;
    std::memset(v3, 0, sizeof *v3);
    std::memcpy(v3, sc, offsetof(rt_scene_desc, meshes));
    v3->struct_size = sizeof *v3;
    v3->abi_version = RT_B200_ABI_VERSION;
    return v3;
}

// The scene is replicated: one host thread per device (the host BVH build is repeated per device -- milliseconds for
// scenes below the device-build threshold; above it every device builds its own tree from the same input)
static int on_every_device(rt_ctx* ctx, int (*fn)(DevCtx*, const rt_scene_desc*), const rt_scene_desc* sc) {
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], fn(ctx->dev[0], sc));
    std::vector<int> rcs(ctx->dev.size(), RT_OK);
    std::vector<std::thread> pool;
    for (size_t i = 1; i < ctx->dev.size(); i++) pool.emplace_back([&, i]() { rcs[i] = fn(ctx->dev[i], sc); });
    rcs[0] = fn(ctx->dev[0], sc);
    for (auto& t : pool) t.join();
    for (size_t i = 0; i < ctx->dev.size(); i++)
        if (rcs[i] != RT_OK) return fwd(ctx, ctx->dev[i], rcs[i]);
    return RT_OK;
}

extern "C" int rt_upload_scene(rt_ctx* ctx, const rt_scene_desc* sc) {
    RT_NEED(ctx);
    rt_scene_desc v3;
    ctx->rendered = false;
    return on_every_device(ctx, dev_upload_scene, widen_v3(sc, &v3));
}

extern "C" int rt_refit_scene(rt_ctx* ctx, const rt_scene_desc* sc) {
    RT_NEED(ctx);
    rt_scene_desc v3;
    const int rc = on_every_device(ctx, dev_refit_scene, widen_v3(sc, &v3));
    if (rc == RT_OK) ctx->rendered = false;  // like an upload; a refused refit changes nothing
    return rc;
}

extern "C" int rt_set_bvh_builder(rt_ctx* ctx, int32_t mode) {
    RT_NEED(ctx);
    for (DevCtx* d : ctx->dev) {
        int rc = dev_set_bvh_builder(d, mode);
        if (rc != RT_OK) return fwd(ctx, d, rc);
    }
    return RT_OK;
}
extern "C" int rt_set_bvh_width(rt_ctx* ctx, int32_t width) {
    RT_NEED(ctx);
    for (DevCtx* d : ctx->dev) {
        int rc = dev_set_bvh_width(d, width);
        if (rc != RT_OK) return fwd(ctx, d, rc);
    }
    return RT_OK;
}

extern "C" int rt_bind_accum(rt_ctx* ctx, void* device_ptr, size_t bytes, int32_t width, int32_t height) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_bind_accum: single-device contexts only (a multi-device context gathers its own frame)");
    return fwd(ctx, ctx->dev[0], dev_bind_accum(ctx->dev[0], device_ptr, bytes, width, height));
}
extern "C" int rt_accum_buffer(rt_ctx* ctx, void** device_ptr, size_t* bytes) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_accum_buffer: single-device contexts only");
    return fwd(ctx, ctx->dev[0], dev_accum_buffer(ctx->dev[0], device_ptr, bytes));
}

// ---- caller-defined cameras ----------------------------------------------------------------------------------------
extern "C" int rt_set_camera_rays(rt_ctx* ctx, const rt_camera_ray* rays, int32_t width, int32_t height) {
    RT_NEED(ctx);
    if (rays) {  // everything is checked before any device changes
        if (width <= 0 || height <= 0 || (long long)width * height >= (1ll << 31))
            return failx(ctx, RT_ERR_INVALID, "rt_set_camera_rays: bad frame size %dx%d", width, height);
        const size_t n = (size_t)width * height;
        auto finite = [](const float* v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); };
        for (size_t k = 0; k < n; k++) {
            const rt_camera_ray& r = rays[k];
            const char* bad = !(finite(r.origin) && finite(r.direction) && finite(r.dx) && finite(r.dy)) ? "a non-finite value"
                              : (r.direction[0] == 0.0f && r.direction[1] == 0.0f && r.direction[2] == 0.0f) ? "a zero direction"
                                                                                                            : nullptr;
            if (bad)
                return failx(ctx, RT_ERR_INVALID, "rt_set_camera_rays: record %zu (pixel %d, %d) has %s", k, (int)(k % (size_t)width),
                             (int)(k / (size_t)width), bad);
        }
    }
    for (DevCtx* d : ctx->dev) {
        const int rc = dev_set_camera_rays(d, rays, width, height);
        if (rc == RT_OK) continue;
        fwd(ctx, d, rc);
        for (DevCtx* e : ctx->dev) dev_set_camera_rays(e, nullptr, 0, 0);  // no device keeps rays the others lack
        return rc;
    }
    return RT_OK;
}

// ---- environment lighting ----------------------------------------------------------------------------------------
extern "C" int rt_set_environment(rt_ctx* ctx, const rt_environment* env) {
    RT_NEED(ctx);
    std::vector<float4> map;
    if (env) {  // everything is checked before any device changes
        if (!env->rgb) return failx(ctx, RT_ERR_INVALID, "rt_set_environment: rgb is NULL");
        if (env->width < 1 || env->height < 1 || (long long)env->width * env->height >= (1ll << 31))
            return failx(ctx, RT_ERR_INVALID, "rt_set_environment: bad map size %dx%d", env->width, env->height);
        const double* R = env->rotation;
        for (int i = 0; i < 9; i++)
            if (!std::isfinite(R[i])) return failx(ctx, RT_ERR_INVALID, "rt_set_environment: rotation[%d] is not finite", i);
        for (int i = 0; i < 3; i++)
            for (int j = i; j < 3; j++) {
                const double dot = R[3 * i] * R[3 * j] + R[3 * i + 1] * R[3 * j + 1] + R[3 * i + 2] * R[3 * j + 2];
                if (std::fabs(dot - (i == j ? 1.0 : 0.0)) > 1e-6)
                    return failx(ctx, RT_ERR_INVALID, "rt_set_environment: the rotation is not orthonormal (rows %d and %d: dot %.9g)", i, j, dot);
            }
        const double det = R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) + R[2] * (R[3] * R[7] - R[4] * R[6]);
        if (std::fabs(det - 1.0) > 1e-6) return failx(ctx, RT_ERR_INVALID, "rt_set_environment: the rotation has determinant %.9g, not +1", det);
        const size_t n = (size_t)env->width * env->height;
        map.resize(kEnvHeader + n);
        for (size_t k = 0; k < n; k++) {
            const float* c = env->rgb + 3 * k;
            for (int i = 0; i < 3; i++)
                if (!(std::isfinite(c[i]) && c[i] >= 0.0f))
                    return failx(ctx, RT_ERR_INVALID, "rt_set_environment: texel %zu (%d, %d) channel %d is %g (texels are finite and >= 0)", k,
                                 (int)(k % (size_t)env->width), (int)(k / (size_t)env->width), i, (double)c[i]);
            map[kEnvHeader + k] = make_float4(c[0], c[1], c[2], 0.0f);
        }
        for (int i = 0; i < 3; i++) map[i] = make_float4((float)R[3 * i], (float)R[3 * i + 1], (float)R[3 * i + 2], 0.0f);
        std::memcpy(&map[0].w, &env->width, 4);
        std::memcpy(&map[1].w, &env->height, 4);
    }
    for (DevCtx* d : ctx->dev) {
        const int rc = dev_set_environment(d, env ? map.data() : nullptr, map.size());
        if (rc == RT_OK) continue;
        fwd(ctx, d, rc);
        for (DevCtx* e : ctx->dev) dev_set_environment(e, nullptr, 0);  // no device keeps a map the others lack
        return rc;
    }
    return RT_OK;
}

// ---- multi-device render ----------------------------------------------------------------------------------------
static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

extern "C" int rt_render(rt_ctx* ctx, const rt_render_params* p) {
    RT_NEED(ctx);
    const int n = (int)ctx->dev.size();
    if (n == 1) return fwd(ctx, ctx->dev[0], dev_render(ctx->dev[0], p));
    if (!p || p->struct_size != sizeof(rt_render_params)) return failx(ctx, RT_ERR_INVALID, "rt_render: bad params struct");
    if (p->width <= 0 || p->height <= 0 || p->samples_per_pixel <= 0) return failx(ctx, RT_ERR_INVALID, "rt_render: width/height/samples must be positive");
    if (p->stream) return failx(ctx, RT_ERR_INVALID, "rt_render: a multi-device context launches on its own streams (stream must be NULL)");
    if (p->flags & RT_FLAG_COMPACT_TILES) return failx(ctx, RT_ERR_INVALID, "rt_render: RT_FLAG_COMPACT_TILES is chosen by a multi-device context itself");
    // the caller's own sharding (several boxes) composes with the devices of this context
    const int ucount = p->shard_count <= 1 ? 1 : p->shard_count, urank = ucount == 1 ? 0 : p->shard_rank;
    if (urank < 0 || urank >= ucount) return failx(ctx, RT_ERR_INVALID, "rt_render: shard_rank %d outside [0,%d)", urank, ucount);
    const int count = ucount * n;
    const int tile = tile_size_of(p);
    const int mode = shard_mode_of(p->width, p->height, tile, count, p->shard_mode);
    if (mode != RT_SHARD_TILES && mode != RT_SHARD_SAMPLES) return failx(ctx, RT_ERR_INVALID, "rt_render: unknown shard_mode %d", p->shard_mode);
    const bool compact = mode == RT_SHARD_TILES && is_pow2(tile);
    rt_render_params q = *p;
    q.shard_mode = mode;
    q.shard_count = count;
    q.tile_size = tile;
    q.flags = (p->flags | RT_FLAG_ASYNC | (compact ? RT_FLAG_COMPACT_TILES : 0u));
    if ((p->flags & RT_FLAG_ACCUMULATE) && ctx->rendered &&
        (ctx->last.width != p->width || ctx->last.height != p->height || ctx->last.shard_mode != mode || ctx->last.tile_size != tile ||
         ctx->last.shard_count != count || ctx->last.shard_rank != urank))
        return failx(ctx, RT_ERR_STATE, "rt_render: RT_FLAG_ACCUMULATE onto a frame of another size or sharding");
    if (!(p->flags & RT_FLAG_ACCUMULATE) && ctx->base_sums) {  // a fresh frame forgets the restored checkpoint
        cudaSetDevice(ctx->dev[0]->device);
        ctx->base_sums.release();
    }
    // every device gets its shard and starts; nothing waits until all are running
    for (int d = 0; d < n; d++) {
        q.shard_rank = urank * n + d;
        int rc = dev_render(ctx->dev[d], &q);
        if (rc != RT_OK) return fwd(ctx, ctx->dev[d], rc);
    }
    ctx->last = q;
    ctx->last.shard_rank = urank;
    ctx->rendered = true;
    if (p->flags & RT_FLAG_ASYNC) return RT_OK;
    for (int d = 0; d < n; d++) {
        int rc = dev_wait(ctx->dev[d]);
        if (rc != RT_OK) return fwd(ctx, ctx->dev[d], rc);
    }
    return RT_OK;
}

// ---- multi-view batches: single-device contexts ------------------------------------------------------------------------
extern "C" int rt_render_views(rt_ctx* ctx, const rt_render_params* params, const rt_camera* cameras, const uint64_t* seeds, int32_t n_views) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_render_views: single-device contexts only");
    return fwd(ctx, ctx->dev[0], dev_render_views(ctx->dev[0], params, cameras, seeds, n_views));
}
extern "C" int rt_download_views(rt_ctx* ctx, int32_t total_spp, int32_t first, int32_t count, float* rgb_linear, uint8_t* rgb8) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_download_views: single-device contexts only");
    return fwd(ctx, ctx->dev[0], dev_download_views(ctx->dev[0], total_spp, first, count, rgb_linear, rgb8));
}

extern "C" int rt_join(rt_ctx* ctx, void* stream) {
    RT_NEED(ctx);
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], dev_join(ctx->dev[0], (cudaStream_t)stream));
    if (stream) return failx(ctx, RT_ERR_INVALID, "rt_join: a multi-device context joins into its own streams (stream must be NULL)");
    for (DevCtx* d : ctx->dev) {
        int rc = dev_join(d, nullptr);
        if (rc != RT_OK) return fwd(ctx, d, rc);
    }
    return RT_OK;
}

extern "C" int rt_sync(rt_ctx* ctx) {
    RT_NEED(ctx);
    for (DevCtx* d : ctx->dev) {
        int rc = dev_sync(d);
        if (rc != RT_OK) return fwd(ctx, d, rc);
    }
    return RT_OK;
}

// src[d] (on device d, `bytes[d]` bytes, produced on that device's stream) -> gather + d * stride on device 0.
// NCCL: one group of n - 1 send/recv pairs over NVLink; otherwise peer copies on the source devices' streams.
static int gather_to_dev0(rt_ctx* ctx, const std::vector<const void*>& src, const std::vector<size_t>& bytes, size_t stride) {
    const int n = (int)ctx->dev.size();
    DevCtx* d0 = ctx->dev[0];
    cudaSetDevice(d0->device);
    if (ctx->gather.reserve(stride * n) != cudaSuccess)
        return failx(ctx, RT_ERR_NOMEM, "cannot allocate %zu bytes of gather staging on device %d", stride * n, d0->device);
    ctx->gathers++;
    if (ctx->gather_mode == 1) {
        // device 0's own part is a local copy; the others travel as send/recv pairs
        cudaSetDevice(d0->device);
        CUX(ctx, cudaMemcpyAsync(ctx->gather, src[0], bytes[0], cudaMemcpyDeviceToDevice, d0->stream));
        int e = ctx->nccl.GroupStart();
        for (int d = 1; d < n && e == 0; d++) {
            if (bytes[d] == 0) continue;
            e = ctx->nccl.Recv(ctx->gather + d * stride, bytes[d], kNcclUint8, d, ctx->comms[0], d0->stream);
            if (e == 0) e = ctx->nccl.Send(src[d], bytes[d], kNcclUint8, 0, ctx->comms[d], ctx->dev[d]->stream);
        }
        const int e2 = ctx->nccl.GroupEnd();
        if (e == 0) e = e2;
        if (e != 0) return failx(ctx, RT_ERR_CUDA, "NCCL gather: %s", ctx->nccl.GetErrorString ? ctx->nccl.GetErrorString(e) : "error");
        for (int d = 1; d < n; d++) {
            cudaSetDevice(ctx->dev[d]->device);
            CUX(ctx, cudaStreamSynchronize(ctx->dev[d]->stream));
        }
        cudaSetDevice(d0->device);
        CUX(ctx, cudaStreamSynchronize(d0->stream));
        return RT_OK;
    }
    for (int d = 0; d < n; d++) {
        if (bytes[d] == 0) continue;
        cudaSetDevice(ctx->dev[d]->device);
        CUX(ctx, cudaMemcpyPeerAsync(ctx->gather + d * stride, d0->device, src[d], ctx->dev[d]->device, bytes[d], ctx->dev[d]->stream));
    }
    for (int d = 0; d < n; d++) {
        cudaSetDevice(ctx->dev[d]->device);
        CUX(ctx, cudaStreamSynchronize(ctx->dev[d]->stream));
    }
    cudaSetDevice(d0->device);
    return RT_OK;
}

// Every pixel of the frame lives on one device: tile shards of this context only, no restored checkpoint to add
static bool one_device_per_pixel(const rt_ctx* ctx) {
    return ctx->dev[0]->frame.layout.compact && !ctx->base_sums && ctx->last.shard_count == (int)ctx->dev.size();
}

// What a device contributes to a gather: its raw sums, or its slots resolved, turned into variance or its AOV sums
// resolved on the device
enum class Plane { Sums, Rgb8, Linear, Variance, Aov };

// The plane of every device's slots, produced on that device and gathered on device 0 (device d at ctx->gather + d * *stride)
static int gather_plane(rt_ctx* ctx, Plane what, int32_t total_spp, size_t* stride) {
    const int n = (int)ctx->dev.size();
    const size_t bpp = what == Plane::Sums || what == Plane::Aov ? 32 : what == Plane::Rgb8 ? 3 : 12;
    const bool resolve = what == Plane::Rgb8 || what == Plane::Linear;
    std::vector<const void*> src((size_t)n);
    std::vector<size_t> bytes((size_t)n);
    *stride = 0;
    for (int d = 0; d < n; d++) {
        DevCtx* dc = ctx->dev[d];
        const size_t slots = dc->frame.layout.slots();
        int rc = what == Plane::Variance ? companion_ready(dc, kMoments, "rt_download_variance")
                 : what == Plane::Aov    ? companion_ready(dc, kAov, "rt_download_aov")
                                         : dev_wait(dc);
        if (rc == RT_OK && what == Plane::Variance) rc = dev_variance_into(dc, total_spp);
        const void* aov_plane = nullptr;
        if (rc == RT_OK && what == Plane::Aov) rc = dev_aov_into(dc, total_spp, 0, &aov_plane);
        if (rc == RT_OK && resolve) rc = stage_buffers(dc, slots, 0);
        if (rc == RT_OK && resolve)
            rc = dev_resolve_into(dc, dc->frame.sums, slots, total_spp, what == Plane::Linear ? dc->out_lin.get() : nullptr, what == Plane::Rgb8 ? dc->out_rgb8.get() : nullptr);
        if (rc != RT_OK) return fwd(ctx, dc, rc);
        src[d] = what == Plane::Sums ? (const void*)dc->frame.sums : what == Plane::Aov ? aov_plane : what == Plane::Rgb8 ? (const void*)dc->out_rgb8 : (const void*)dc->out_lin;
        bytes[d] = slots * bpp;
        *stride = std::max(*stride, (bytes[d] + 255) & ~(size_t)255);
    }
    return gather_to_dev0(ctx, src, bytes, *stride);
}

// The sums of all devices as ONE full row-major frame on device 0 (in d0->frame_scratch): compact tiles are
// gathered and scattered, sample-sharded full frames are added; a restored checkpoint is added on top.
static int gather_sums_full(rt_ctx* ctx) {
    const int n = (int)ctx->dev.size();
    DevCtx* d0 = ctx->dev[0];
    const int w = ctx->last.width, h = ctx->last.height;
    const size_t full = (size_t)w * h * 32;
    size_t stride = 0;
    int rc = gather_plane(ctx, Plane::Sums, 0, &stride);
    if (rc != RT_OK) return rc;
    cudaSetDevice(d0->device);
    rc = stage_buffers(d0, 0, full);
    if (rc != RT_OK) return fwd(ctx, d0, rc);
    if (d0->frame.layout.compact) {
        // the devices hold shards urank * n + d of count ucount * n: inside this context they are n consecutive shards, so
        // the scatter works on the sub-frame "tiles with t mod count in [urank * n, urank * n + n)"; with ucount == 1
        // (the only case a single box needs) that is every tile
        if (ctx->last.shard_count != n) return failx(ctx, RT_ERR_UNSUPPORTED, "gathering a frame that is also sharded across contexts: download the shards (rt_resolve_tiles) instead");
        CUX(ctx, launch_untile(32, ctx->gather, stride, n, -1, w, h, ctx->last.tile_size, d0->frame_scratch, d0->stream));
    } else {
        CUX(ctx, cudaMemcpyAsync(d0->frame_scratch, ctx->gather, full, cudaMemcpyDeviceToDevice, d0->stream));
        const size_t words = full / 8;
        for (int d = 1; d < n; d++)
            add_sums_kernel<<<(unsigned)((words + 255) / 256), 256, 0, d0->stream>>>((unsigned long long*)d0->frame_scratch.get(),
                                                                                     (const unsigned long long*)(ctx->gather + d * stride), words);
    }
    if (ctx->base_sums && ctx->base_w == w && ctx->base_h == h) {
        const size_t words = full / 8;
        add_sums_kernel<<<(unsigned)((words + 255) / 256), 256, 0, d0->stream>>>((unsigned long long*)d0->frame_scratch.get(), ctx->base_sums, words);
    }
    CUX(ctx, cudaGetLastError());
    return RT_OK;
}

extern "C" int rt_download(rt_ctx* ctx, int32_t total_spp, float* rgb_linear, uint8_t* rgb8) {
    RT_NEED(ctx);
    const int n = (int)ctx->dev.size();
    if (n == 1) return fwd(ctx, ctx->dev[0], dev_download(ctx->dev[0], total_spp, rgb_linear, rgb8));
    if (!ctx->rendered) return failx(ctx, RT_ERR_STATE, "rt_download: nothing rendered yet");
    if (total_spp <= 0) return failx(ctx, RT_ERR_INVALID, "rt_download: total_spp must be positive");
    if (!rgb_linear && !rgb8) return RT_OK;
    DevCtx* d0 = ctx->dev[0];
    const int w = ctx->last.width, h = ctx->last.height;
    if (!one_device_per_pixel(ctx)) {
        // sums first (sample-sharded frames, restored checkpoints), then one resolve of the whole frame on device 0
        int rc = gather_sums_full(ctx);
        if (rc != RT_OK) return rc;
        return fwd(ctx, d0, resolve_to_host(d0, (const unsigned long long*)d0->frame_scratch.get(), AccumLayout{w, h}, total_spp, rgb_linear, rgb8));
    }
    // tiles: resolve where they were rendered, move 3 (RGB8) or 12 (float) bytes per pixel instead of 32
    for (int pass = 0; pass < 2; pass++) {
        const bool lin = pass == 1;
        if ((lin && !rgb_linear) || (!lin && !rgb8)) continue;
        size_t stride = 0;
        int rc = gather_plane(ctx, lin ? Plane::Linear : Plane::Rgb8, total_spp, &stride);
        if (rc != RT_OK) return rc;
        rc = dev_untile(d0, ctx->gather, stride, lin ? 12 : 3, n, w, h, ctx->last.tile_size, lin ? (void*)rgb_linear : (void*)rgb8);
        if (rc != RT_OK) return fwd(ctx, d0, rc);
    }
    return RT_OK;
}

extern "C" int rt_accum_download(rt_ctx* ctx, uint64_t* host, size_t bytes) {
    RT_NEED(ctx);
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], dev_accum_download(ctx->dev[0], host, bytes));
    if (!host) return RT_ERR_INVALID;
    if (!ctx->rendered) return failx(ctx, RT_ERR_STATE, "rt_accum_download: nothing rendered yet");
    const size_t full = (size_t)ctx->last.width * ctx->last.height * 32;
    if (bytes < full) return failx(ctx, RT_ERR_INVALID, "rt_accum_download: need %zu bytes, got %zu", full, bytes);
    int rc = gather_sums_full(ctx);
    if (rc != RT_OK) return rc;
    return fwd(ctx, ctx->dev[0], plane_to_host(ctx->dev[0], ctx->dev[0]->frame_scratch, 32, AccumLayout{ctx->last.width, ctx->last.height}, host));
}

extern "C" int rt_accum_upload(rt_ctx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height) {
    RT_NEED(ctx);
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], dev_accum_upload(ctx->dev[0], host, bytes, width, height));
    if (!host) return RT_ERR_INVALID;
    if (width <= 0 || height <= 0 || (long long)width * height >= (1ll << 31)) return failx(ctx, RT_ERR_INVALID, "rt_accum_upload: bad frame size %dx%d", width, height);
    const size_t need = (size_t)width * height * 32;
    if (bytes != need) return failx(ctx, RT_ERR_INVALID, "rt_accum_upload: a %dx%d frame is %zu bytes, got %zu", width, height, need, bytes);
    // The restored sums stay a full frame on device 0 and are added when the frame is gathered; the devices start their
    // (compact) buffers from zero: sums are associative, so the result is the uninterrupted render's, bit for bit.
    DevCtx* d0 = ctx->dev[0];
    for (DevCtx* d : ctx->dev) {
        int rc = dev_wait(d);
        if (rc != RT_OK) return fwd(ctx, d, rc);
        // forget what the devices hold: the next RT_FLAG_ACCUMULATE render starts from cleared buffers
        cudaSetDevice(d->device);
        if (d->frame.sums) CUX(ctx, cudaMemsetAsync(d->frame.sums, 0, d->frame.sums_bytes(), d->stream));
        CUX(ctx, cudaStreamSynchronize(d->stream));
        frame_forget(d);  // companions are not restored across devices (rt_moments_upload is single-device)
    }
    cudaSetDevice(d0->device);
    ctx->base_sums.release();  // allocated for exactly this frame
    if (ctx->base_sums.reserve(need) != cudaSuccess) return failx(ctx, RT_ERR_NOMEM, "rt_accum_upload: cannot allocate %zu bytes", need);
    ctx->base_w = width;
    ctx->base_h = height;
    CUX(ctx, cudaMemcpyAsync(ctx->base_sums, host, need, cudaMemcpyHostToDevice, d0->stream));
    CUX(ctx, cudaStreamSynchronize(d0->stream));
    return RT_OK;
}

// ---- second moments (RT_FLAG_MOMENTS) and auxiliary outputs (RT_FLAG_AOV) --------------------------------------------
// A multi-device frame has per-device variance and AOVs only when each pixel lives on one device: tiles, no restored
// checkpoint.
static int multi_per_pixel_frame(rt_ctx* ctx, const char* what) {
    if (!ctx->rendered) return failx(ctx, RT_ERR_STATE, "%s: nothing rendered yet", what);
    if (!one_device_per_pixel(ctx))
        return failx(ctx, RT_ERR_UNSUPPORTED, "%s: a multi-device context resolves tile-sharded frames without a restored checkpoint only", what);
    return RT_OK;
}

// A companion's plane of a multi-device frame (`what` names the entry point), produced where the tiles were rendered and
// gathered at `bpp` bytes per pixel: the variance like the linear radiance of rt_download, the AOVs resolved
static int download_companion(rt_ctx* ctx, Plane plane, int bpp, const char* what, int32_t total_spp, float* host) {
    int rc = multi_per_pixel_frame(ctx, what);
    if (rc != RT_OK) return rc;
    size_t stride = 0;
    rc = gather_plane(ctx, plane, total_spp, &stride);
    if (rc != RT_OK) return rc;
    return fwd(ctx, ctx->dev[0], dev_untile(ctx->dev[0], ctx->gather, stride, bpp, (int)ctx->dev.size(), ctx->last.width, ctx->last.height, ctx->last.tile_size, host));
}

extern "C" int rt_download_variance(rt_ctx* ctx, int32_t total_spp, float* variance) {
    RT_NEED(ctx);
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], dev_download_variance(ctx->dev[0], total_spp, variance));
    if (!variance) return RT_ERR_INVALID;
    if (total_spp < 2) return failx(ctx, RT_ERR_INVALID, "rt_download_variance: total_spp must be at least 2");
    return download_companion(ctx, Plane::Variance, 12, "rt_download_variance", total_spp, variance);
}

extern "C" int rt_download_aov(rt_ctx* ctx, int32_t total_spp, float* aov) {
    RT_NEED(ctx);
    if (ctx->dev.size() == 1) return fwd(ctx, ctx->dev[0], dev_download_aov(ctx->dev[0], total_spp, aov));
    if (!aov) return RT_ERR_INVALID;
    if (total_spp <= 0) return failx(ctx, RT_ERR_INVALID, "rt_download_aov: total_spp must be positive");
    return download_companion(ctx, Plane::Aov, 32, "rt_download_aov", total_spp, aov);
}

extern "C" int rt_frame_noise(rt_ctx* ctx, int32_t total_spp, double* mean_radiance, double* rms_std_error) {
    RT_NEED(ctx);
    if (!mean_radiance || !rms_std_error) return RT_ERR_INVALID;
    if (total_spp < 2) return failx(ctx, RT_ERR_INVALID, "rt_frame_noise: total_spp must be at least 2");
    if (ctx->dev.size() > 1) {
        int rc = multi_per_pixel_frame(ctx, "rt_frame_noise");
        if (rc != RT_OK) return rc;
    }
    // integer partials of every device added on the host: the same words whatever the device count
    uint64_t sum[12] = {0}, pixels = 0;
    for (DevCtx* d : ctx->dev) {
        uint64_t part[12], px = 0;
        int rc = dev_noise_partials(d, total_spp, part, &px);
        if (rc != RT_OK) return fwd(ctx, d, rc);
        for (int k = 0; k < 12; k++) sum[k] += part[k];
        pixels += px;
    }
    noise_from_partials(sum, pixels, total_spp, mean_radiance, rms_std_error);
    return RT_OK;
}

extern "C" int rt_moments_download(rt_ctx* ctx, uint64_t* host, size_t bytes) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_moments_download: single-device contexts only");
    return fwd(ctx, ctx->dev[0], dev_moments_download(ctx->dev[0], host, bytes));
}

extern "C" int rt_moments_upload(rt_ctx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_moments_upload: single-device contexts only");
    return fwd(ctx, ctx->dev[0], dev_moments_upload(ctx->dev[0], host, bytes, width, height));
}

extern "C" int rt_resolve_tiles(rt_ctx* ctx, int32_t total_spp, float* dev_rgb_linear, uint8_t* dev_rgb8, size_t capacity_pixels) {
    RT_NEED(ctx);
    if (ctx->dev.size() != 1) return failx(ctx, RT_ERR_UNSUPPORTED, "rt_resolve_tiles: single-device contexts only (a multi-device context gathers in rt_download)");
    return fwd(ctx, ctx->dev[0], dev_resolve_tiles(ctx->dev[0], total_spp, dev_rgb_linear, dev_rgb8, capacity_pixels));
}

extern "C" int rt_untile(rt_ctx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count, int32_t width,
                         int32_t height, int32_t tile_size, void* host_out) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_untile(ctx->dev[0], dev_shards, shard_stride_bytes, bytes_per_pixel, shard_count, width, height, tile_size, host_out));
}

// ---- asynchronous hand-out: the copy to (pinned) host memory overlaps the next pass ------------------------------------
extern "C" int rt_download_begin(rt_ctx* ctx, int32_t total_spp, int32_t want_linear, int32_t want_rgb8) {
    RT_NEED(ctx);
    const int n = (int)ctx->dev.size();
    if (n == 1) return fwd(ctx, ctx->dev[0], dev_download_begin(ctx->dev[0], total_spp, want_linear, want_rgb8));
    // several devices: the gather is synchronous (it is microseconds over NVLink), the PCIe copy is what overlaps
    if (!ctx->rendered) return failx(ctx, RT_ERR_STATE, "rt_download_begin: nothing rendered yet");
    if (total_spp <= 0 || (!!want_linear == !!want_rgb8)) return failx(ctx, RT_ERR_INVALID, "rt_download_begin: a multi-device context hands out ONE of linear / rgb8 per call");
    if (!one_device_per_pixel(ctx))
        return failx(ctx, RT_ERR_UNSUPPORTED, "rt_download_begin: tile-sharded frames without a restored checkpoint only (use rt_download)");
    const bool lin = want_linear != 0;
    size_t stride = 0;
    int rc = gather_plane(ctx, lin ? Plane::Linear : Plane::Rgb8, total_spp, &stride);
    if (rc != RT_OK) return rc;
    return fwd(ctx, ctx->dev[0], dev_untile_begin(ctx->dev[0], ctx->gather, stride, lin ? 12 : 3, n, ctx->last.width, ctx->last.height, ctx->last.tile_size));
}
extern "C" int rt_untile_begin(rt_ctx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count,
                               int32_t width, int32_t height, int32_t tile_size) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_untile_begin(ctx->dev[0], dev_shards, shard_stride_bytes, bytes_per_pixel, shard_count, width, height, tile_size));
}
extern "C" int rt_frame_end(rt_ctx* ctx, const float** rgb_linear, const uint8_t** rgb8) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_frame_end(ctx->dev[0], rgb_linear, rgb8));
}

extern "C" int rt_render_aov(rt_ctx* ctx, int32_t width, int32_t height, int32_t* prim_id, float* t, float* normal, float* point, float* uv) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_render_aov(ctx->dev[0], width, height, prim_id, t, normal, point, uv));
}

extern "C" int rt_get_stats(rt_ctx* ctx, rt_stats* out) {
    RT_NEED(ctx);
    if (!out) return RT_ERR_INVALID;
    int rc = dev_get_stats(ctx->dev[0], out);
    if (rc != RT_OK) return fwd(ctx, ctx->dev[0], rc);
    out->devices = (uint32_t)ctx->dev.size();
    out->gather_mode = ctx->dev.size() > 1 ? (uint32_t)(ctx->gather_mode + 1) : 0u;
    for (size_t i = 1; i < ctx->dev.size(); i++) {
        const rt_stats& s = ctx->dev[i]->stats;
        out->render_ms = std::max(out->render_ms, s.render_ms);  // the devices run concurrently
        out->upload_ms = std::max(out->upload_ms, s.upload_ms);
        out->samples += s.samples;
        out->rays += s.rays;
        out->node_visits += s.node_visits;
        out->box_tests += s.box_tests;
        out->sphere_tests += s.sphere_tests;
        out->quad_tests += s.quad_tests;
        out->triangle_tests += s.triangle_tests;
        out->medium_queries += s.medium_queries;
        out->boundary_tests += s.boundary_tests;
        out->fp64_sphere_tests += s.fp64_sphere_tests;
        out->nonfinite_samples += s.nonfinite_samples;
        out->empty_node_steps += s.empty_node_steps;
        out->kernel_launches += s.kernel_launches;
        out->blocks += s.blocks;
    }
    return RT_OK;
}

extern "C" int rt_measure_fp32_peak(rt_ctx* ctx, double* tflops) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_measure_fp32_peak(ctx->dev[0], tflops));
}
extern "C" int rt_measure_l1_peak(rt_ctx* ctx, double* gbs) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_measure_l1_peak(ctx->dev[0], gbs));
}
extern "C" int rt_probe_texture(rt_ctx* ctx, int32_t texture, int32_t n, const float* uvp, float* rgb) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_probe_texture(ctx->dev[0], texture, n, uvp, rgb));
}
extern "C" int rt_probe_scatter(rt_ctx* ctx, int32_t material, int32_t n, const float* in_rec, const float* uniforms, float* out_rec) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_probe_scatter(ctx->dev[0], material, n, in_rec, uniforms, out_rec));
}
extern "C" int rt_probe_hit(rt_ctx* ctx, int32_t n, const float* rays, int32_t* prim_id, float* t, float* normal, float* uv) {
    RT_NEED(ctx);
    return fwd(ctx, ctx->dev[0], dev_probe_hit(ctx->dev[0], n, rays, prim_id, t, normal, uv));
}
