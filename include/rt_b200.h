/*
 * rt_b200.h — C ABI of the B200-native path-tracing core (librt_b200.so).
 *
 * This is the drop-in boundary that sits UNDER the reference's
 *     void camera::render(const hittable& world, std::vector<point_light>& lights)
 * (reference Camera.txt:54, called from main.cpp:471 after main.cpp:442 wrapped the
 * world in a bvh_node).  The reference has no FFI of its own; a host program keeps
 * building the same make_shared<sphere/quad/triangle/...> object graph, and the
 * host-side mirror of the scene API (raytracingoneweekendapplication_b200/host/)
 * flattens that graph once into the plain-old-data arrays declared here and makes
 * the three calls rt_upload_scene / rt_render / rt_download.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no C++ or torch types.
 *   - every function returns RT_OK (0) or a non-zero rt_status; the message of the
 *     last failure on a context is available from rt_last_error().
 *   - nothing throws across the boundary; there is no global state.
 *   - a context is driven by one host thread at a time; distinct contexts are
 *     independent.  A context owns one GPU or several GPUs of one box (rt_create);
 *     under torchrun every process creates a one-GPU context and shards the frame with
 *     rt_render_params::shard_rank / shard_count.
 *   - all pointers passed IN are copied before the call returns (the caller keeps
 *     ownership and may free immediately); all pointers passed OUT are
 *     caller-allocated.
 *   - there is NO CPU fallback: without a CUDA device rt_create fails with
 *     RT_ERR_CUDA.
 *
 * Geometry and colours cross the boundary as double (the reference's arithmetic
 * type, vec3.h:9); the device path computes in FP32, with an FP64 sphere test for
 * rays that start very close to a large sphere (DESIGN.md "precision").
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 4

typedef struct rt_ctx rt_ctx;

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = 1,     /* bad argument / malformed scene description   */
    RT_ERR_CUDA = 2,        /* CUDA runtime error, or no usable device       */
    RT_ERR_NOMEM = 3,       /* host or device allocation failed              */
    RT_ERR_STATE = 4,       /* call order violated (e.g. render before upload) */
    RT_ERR_UNSUPPORTED = 5, /* feature outside the hot path                  */
    RT_ERR_KERNEL = 6       /* device-side guard tripped (reserved: the traversal stack depth is checked at upload) */
} rt_status;

/* ---------------------------------------------------------------------------
 * Scene description (what the flatten step of the host mirror produces).
 * ------------------------------------------------------------------------- */

/* Rigid instance transform p_world = R * p_obj + t, R row-major.  Replaces the
 * reference's translate / rotate_y wrapper chain (hittable.h:39-65, 67-146);
 * xform index -1 means identity.  rt_upload_scene bakes it into the geometry. */
typedef struct rt_xform {
    double r[9];
    double t[3];
} rt_xform;

typedef enum rt_prim_type {
    RT_PRIM_SPHERE = 0,   /* sphere.h:9-75 (static and moving)                */
    RT_PRIM_QUAD = 1,     /* quad.h:8-84 (box() = six of these, quad.h:86-108) */
    RT_PRIM_TRIANGLE = 2, /* triangle.h:14-143                                */
    RT_PRIM_MESH = 3      /* all triangles of one rt_mesh (world only, not a medium boundary) */
} rt_prim_type;

typedef struct rt_sphere {
    double center0[3];    /* centre at time 0                                  */
    double center_vec[3]; /* centre(time) = center0 + time * center_vec (sphere.h:33) */
    double radius;
    int32_t material;
    int32_t xform;
} rt_sphere;

typedef struct rt_quad {
    double Q[3], u[3], v[3];
    int32_t material;
    int32_t xform;
} rt_quad;

typedef struct rt_triangle {
    double p0[3], p1[3], p2[3];
    float uv0[2], uv1[2], uv2[2]; /* glm::vec2 in the reference (triangle.h:130-132) */
    int32_t material;
    int32_t xform;
} rt_triangle;

/* An indexed triangle mesh (mesh.h's positions and UVs are floats, so this carries exactly the values a
 * run of rt_triangle records would, in about a fifth of the bytes).  Triangle k has the corners
 * positions[3 * indices[3k + c] ..] for c = 0, 1, 2 and the UVs uvs[2 * uv_indices[3k + c] ..]; with
 * uv_indices NULL the UV index is the position index (then n_uvs == n_vertices), with uvs NULL every
 * triangle gets (0,0), (1,0), (0,1) like the four-argument triangle (triangle.h:24-26).  Several meshes
 * may share the same arrays (e.g. with different xforms).  Every index is checked at upload. */
typedef struct rt_mesh {
    const float* positions;     /* n_vertices x 3                                   */
    const uint32_t* indices;    /* n_triangles x 3                                  */
    const float* uvs;           /* NULL, or n_uvs x 2                               */
    const uint32_t* uv_indices; /* NULL, or n_triangles x 3 (requires uvs)          */
    int32_t n_vertices, n_triangles, n_uvs;
    int32_t material;
    int32_t xform;
    int32_t pad_;
} rt_mesh;

/* A reference to one primitive, or with RT_PRIM_MESH to all triangles of mesh `index`.  Canonical
 * primitive ids (reported by the primary-hit AOV) are assigned in world order: a single primitive
 * takes one id, a mesh ref n_triangles consecutive ids in index-buffer order.  Without meshes the id
 * is the position in rt_scene_desc::world (depth-first insertion order of the scene graph; a box()
 * contributes six consecutive ids). */
typedef struct rt_prim_ref {
    int32_t type;  /* rt_prim_type */
    int32_t index; /* into the typed array */
} rt_prim_ref;

typedef struct rt_medium {
    int32_t boundary_first; /* range in rt_scene_desc::boundary_refs            */
    int32_t boundary_count;
    double density;         /* constant_medium.h:11: neg_inv_density = -1/density */
    int32_t multiplicity;   /* how many times the reference's BVH calls hit() on
                               this object per visit: 2 in a 1-object leaf
                               (bvh.h:31-33), which multiplies the effective density */
    int32_t material;       /* the isotropic phase function (material.h:124-138) */
    int32_t xform;          /* rotates the arbitrary normal (1,0,0) of constant_medium.h:48 */
    int32_t pad_;
} rt_medium;

typedef enum rt_material_type {
    RT_MAT_LAMBERTIAN = 0,     /* material.h:22-41   */
    RT_MAT_METAL = 1,          /* material.h:78-92   */
    RT_MAT_DIELECTRIC = 2,     /* material.h:43-76   */
    RT_MAT_DIFFUSE_LIGHT = 3,  /* material.h:94-104  */
    RT_MAT_EMISSIVE_LIGHT = 4, /* material.h:105-122 */
    RT_MAT_ISOTROPIC = 5,      /* material.h:124-138 */
    RT_MAT_SPECULAR = 6        /* material.h:140-172 */
} rt_material_type;

typedef struct rt_material {
    int32_t type;
    int32_t texture;  /* lambertian / lights / isotropic; -1 otherwise          */
    double albedo[3]; /* metal, specular                                        */
    double param;     /* metal: fuzz; dielectric: refraction_index; specular: shininess */
} rt_material;

typedef enum rt_texture_type {
    RT_TEX_SOLID = 0,            /* texture.h:20-32   */
    RT_TEX_CHECKER = 1,          /* texture.h:34-56   */
    RT_TEX_CHECKER_TRIANGLE = 2, /* texture.h:58-84   */
    RT_TEX_IMAGE = 3,            /* texture.h:86-108  */
    RT_TEX_NOISE = 4             /* texture.h:110-120 */
} rt_texture_type;

typedef struct rt_texture {
    int32_t type;
    int32_t even, odd; /* checker variants: child texture indices               */
    int32_t image;     /* RT_TEX_IMAGE: index into images (-1: no data -> cyan)  */
    int32_t perlin;    /* RT_TEX_NOISE: index into perlins                       */
    int32_t pad_;
    double color[3];   /* RT_TEX_SOLID                                           */
    double scale;      /* checker variants: inv_scale; noise: scale              */
} rt_texture;

/* rtw_image::bdata (rtw_stb_image.h:99-121): 3 bytes per texel, top row first,
 * already linearised (gamma 2.2) and re-quantised by the host loader. */
typedef struct rt_image {
    int32_t width, height;
    const uint8_t* rgb;
} rt_image;

/* perlin.h:52-57, built on the host (its tables come from rand()). */
typedef struct rt_perlin {
    double randvec[256][3];
    int32_t perm_x[256], perm_y[256], perm_z[256];
} rt_perlin;

/* point_light.h:9-28 */
typedef struct rt_point_light {
    double position[3];
    double intensity[3];
    double size;
} rt_point_light;

/* The public camera fields of Camera.txt:39-52 (image size travels in
 * rt_render_params).  camera::initialize (Camera.txt:136-175) runs inside the
 * library. */
typedef struct rt_camera {
    double lookfrom[3], lookat[3], vup[3];
    double vfov;
    double defocus_angle;
    double focus_dist;
    double background[3];
} rt_camera;

typedef struct rt_scene_desc {
    uint32_t struct_size; /* sizeof(rt_scene_desc), for forward compatibility    */
    uint32_t abi_version; /* RT_B200_ABI_VERSION                                 */

    const rt_prim_ref* world; /* every surface leaf of the world in canonical order */
    int32_t n_world;
    const rt_prim_ref* boundary_refs; /* boundaries of the media                 */
    int32_t n_boundary_refs;

    const rt_sphere* spheres;     int32_t n_spheres;
    const rt_quad* quads;         int32_t n_quads;
    const rt_triangle* triangles; int32_t n_triangles;
    const rt_medium* media;       int32_t n_media;
    const rt_xform* xforms;       int32_t n_xforms;

    const rt_material* materials; int32_t n_materials;
    const rt_texture* textures;   int32_t n_textures;
    const rt_image* images;       int32_t n_images;
    const rt_perlin* perlins;     int32_t n_perlins;
    const rt_point_light* lights; int32_t n_lights;

    rt_camera camera;

    /* ABI version 4.  A version-3 caller passes struct_size == offsetof(rt_scene_desc, meshes) and
     * abi_version 3; its scene is read as one without meshes. */
    const rt_mesh* meshes;        int32_t n_meshes;
} rt_scene_desc;

/* ---------------------------------------------------------------------------
 * Rendering
 * ------------------------------------------------------------------------- */

typedef enum rt_shard_mode {
    RT_SHARD_AUTO = 0,    /* tiles when every shard gets >= 256 tiles, else samples */
    RT_SHARD_TILES = 1,   /* interleaved tile_size x tile_size tiles: tile t -> shard t mod count */
    RT_SHARD_SAMPLES = 2  /* sample index s -> shard s mod count                  */
} rt_shard_mode;

#define RT_FLAG_ACCUMULATE 1u /* add to the accumulation buffer instead of clearing it first
                                 (progressive rendering: pass a fresh spp_begin each time)   */
#define RT_FLAG_ASYNC 2u      /* enqueue on `stream` and return; rt_sync() / rt_download wait */
#define RT_FLAG_STATS 4u      /* count rays / node visits / prim tests (slower kernel variant) */
#define RT_FLAG_NEE 8u        /* opt-in next-event estimation: lambertian and isotropic vertices sample the quad
                                 emitters of the scene directly (shadow ray, media transmittance), weighted with the
                                 density of the reference's own direction sampler, so the CONVERGED image is the one
                                 the reference converges to; individual samples differ, noise is lower.  Ignored when
                                 the scene has no quad emitter. */
#define RT_FLAG_COMPACT_TILES 32u /* tile-sharded render (shard_mode RT_SHARD_TILES, tile_size a power of two) into a COMPACT
                                 accumulation buffer that holds only this shard's tiles: tile t of the frame is local tile
                                 t / shard_count of shard t mod shard_count, stored as tile_size x tile_size slots --
                                 1 / shard_count of the frame instead of all of it.  rt_resolve_tiles / rt_untile move and
                                 reassemble such shards; rt_download and rt_accum_download still hand out the full frame
                                 (this shard's tiles in place, zero elsewhere).  A multi-device context sets it itself. */
#define RT_FLAG_SHADOWED_POINT_LIGHTS 16u /* opt-in: a shadow ray (and media transmittance) per point light in the
                                 term of Camera.txt:240-272.  The reference's point lights are unshadowed, so this
                                 changes the image on purpose. */

#define RT_FLAG_OVERLAP 64u   /* with RT_FLAG_ASYNC | RT_FLAG_ACCUMULATE: consecutive passes onto the same frame run on two
                                 internal streams of the context, each with its own work counter, so that the drain of one
                                 pass (its last paths, up to max_depth dependent bounces while most SMs idle: ~1 ms on C5)
                                 overlaps the start of the next.  The sums are order-independent integers, so the frame
                                 is bit-identical to serial passes.  The passes are ordered after what `stream` holds when
                                 rt_render is called; `stream` itself does NOT wait for them: call rt_join (stream order)
                                 or anything that waits (rt_sync, rt_download, rt_resolve_tiles, ...) before using the
                                 frame.  Ignored (a plain asynchronous pass) without both other flags and with
                                 RT_FLAG_STATS.  rt_stats.render_ms is then the average per overlapped pass. */
#define RT_FLAG_MOMENTS 128u  /* also accumulate per-pixel second moments (exact integer sums of the squared samples) into a
                                 moments buffer of the context (48 bytes per pixel, the layout of the sums).  A pass
                                 without RT_FLAG_ACCUMULATE starts them; an accumulating pass with the flag needs a frame
                                 whose moments describe its sums (RT_ERR_STATE otherwise), and one without it leaves the
                                 frame without moments.  Runs the general kernel instances (plain / NEE); with RT_FLAG_STATS
                                 it is RT_ERR_UNSUPPORTED.  The image is the same as without the flag. */
#define RT_FLAG_AOV 256u      /* also add each camera sample's first-vertex albedo, normal, depth and hit to AOV sums of the
                                 context (64 bytes per pixel, the layout of the sums), read with rt_download_aov.  The
                                 state rules are those of RT_FLAG_MOMENTS: a pass without RT_FLAG_ACCUMULATE starts them;
                                 an accumulating pass with the flag needs a frame whose AOV sums describe its sums
                                 (RT_ERR_STATE otherwise); a pass without it, and rt_accum_upload, leave the frame without
                                 them.  Runs the general kernel instances (plain / NEE); with RT_FLAG_STATS or
                                 RT_FLAG_MOMENTS it is RT_ERR_UNSUPPORTED.  The image is the same as without the flag. */
#define RT_FLAG_CAMERA_RAYS 512u /* the primary rays come from the records of rt_set_camera_rays instead of the uploaded
                                 camera (see there).  RT_ERR_STATE without rays, RT_ERR_INVALID when width / height are
                                 not those of the rays; with RT_FLAG_STATS or RT_FLAG_MOMENTS, and in rt_render_views,
                                 RT_ERR_UNSUPPORTED.  Every other flag, shards and multi-device contexts work with it. */

typedef struct rt_render_params {
    uint32_t struct_size;
    int32_t width, height;       /* image_width, image_height (Camera.txt:39,137) */
    int32_t samples_per_pixel;   /* Camera.txt:42: samples traced by this call     */
    int32_t max_depth;           /* Camera.txt:43 */
    int32_t spp_begin;           /* index of the first sample (Philox counter word) */
    uint64_t seed;               /* Philox key; the image is a pure function of
                                    (scene, width, height, sample range, depth, seed)
                                    and does not depend on sharding or scheduling  */
    int32_t tile_size;           /* 0 -> 16 */
    int32_t shard_mode;          /* rt_shard_mode */
    int32_t shard_rank;          /* this context's shard, 0 <= rank < count       */
    int32_t shard_count;         /* 0 or 1: render the whole frame                */
    uint32_t flags;              /* RT_FLAG_*                                     */
    int32_t reserved_;
    void* stream;                /* cudaStream_t to launch on; NULL = the context's own */
} rt_render_params;

typedef struct rt_stats {
    double render_ms;          /* device time of the last synchronous rt_render (CUDA events) */
    double upload_ms;          /* host time of the last rt_upload_scene or rt_refit_scene (incl. BVH build) */
    uint64_t samples;          /* camera samples traced by the last rt_render       */
    uint64_t rays;             /* world.hit root queries incl. primary (RT_FLAG_STATS) */
    uint64_t node_visits;      /* BVH nodes fetched (each holds two child boxes)    */
    uint64_t box_tests;        /* child-box slab tests                             */
    uint64_t sphere_tests, quad_tests, triangle_tests;
    uint64_t medium_queries;   /* constant_medium::hit evaluations                 */
    uint64_t boundary_tests;   /* primitive tests made by those (two passes each)  */
    uint64_t fp64_sphere_tests;/* sphere tests that took the FP64 path             */
    uint64_t nonfinite_samples;/* samples dropped because their radiance was NaN/Inf */
    uint32_t kernel_launches;  /* launches of this library's kernels in the last rt_render */
    uint32_t bvh_nodes;        /* size of the acceleration structure               */
    uint32_t bvh_depth;
    uint32_t bvh_leaves;
    uint32_t regs_per_thread;
    uint32_t threads_per_block, blocks;
    uint32_t local_bytes_per_thread;
    /* lane occupancy of the megakernel's phases (RT_FLAG_STATS): warp-level iterations and the
     * lanes that did work in them -- desc = one BVH node step, leaf = one leaf visit, shade = one
     * shade phase; desc_trav_lanes = lanes holding a ray during a node step (working or waiting) */
    uint64_t desc_iters, desc_lanes, desc_trav_lanes;
    uint64_t leaf_iters, leaf_lanes;
    uint64_t shade_iters, shade_lanes;
    /* shape of a ray's traversal (RT_FLAG_STATS): histograms of the node steps before the first
     * leaf visit [0,64), between two leaf visits [64,128), after the last one [128,192) (last bin
     * of each = that many or more), and of the leaf visits per ray [192,208) */
    uint64_t trav_hist[208];
    /* scene-upload path of the last rt_upload_scene: 1 = acceleration structure and device records
     * built by CUDA kernels, with the device time of the build and of the raw-input copy */
    uint32_t bvh_on_device, reserved_;
    double device_build_ms, device_copy_in_ms;
    double device_top_ms; /* host time of the SAH top levels of the device-built tree (sync + copies included) */
    /* acceleration structure the render kernels traverse: 2 = binary tree of 64-byte nodes, 8 / 4 = wide
     * tree with 8-bit quantised child boxes (80 / 48 bytes per node); node count and levels of the wide tree */
    uint32_t bvh_width, wide_nodes, wide_depth, reserved2_;
    uint64_t empty_node_steps; /* node steps in which no child box was hit (RT_FLAG_STATS) */
    /* multi-device contexts: devices of the context (counters above are summed over them, render_ms is the slowest
     * device's) and how rt_download gathers their tiles on device 0: 0 single device, 1 peer copies, 2 NCCL send/recv */
    uint32_t devices, gather_mode;
    /* last rt_upload_scene or rt_refit_scene: bytes copied to the device, and 1 when the scene was byte-identical to the
     * one already uploaded (same builder settings), so that only the staged arena was copied again -- no validation, no
     * BVH build */
    uint64_t upload_bytes;
    uint32_t scene_reused, reserved3_;
} rt_stats;

/* Create a context on the CUDA devices device_ids[0 .. n_devices).  With n_devices > 1 the context
 * replicates the scene on every device, rt_render gives tile t of the frame to device t mod n_devices
 * (compact per-device tile buffers, all devices running concurrently) and rt_download gathers the resolved
 * tiles on device_ids[0] over NVLink (NCCL send/recv when libnccl.so.2 loads, peer copies otherwise;
 * RT_B200_GATHER=nccl|p2p forces one).  The image does not depend on n_devices, bit for bit.  Replaces the
 * reference's row bands over CPU threads (Camera.txt:59-61, 96-100).  *out is set even on failure so that
 * rt_last_error works; destroy it. */
int rt_create(rt_ctx** out, const int* device_ids, int n_devices);
int rt_device_count(const rt_ctx* ctx);
int rt_visible_devices(void); /* CUDA devices this process can see (0 without a driver); no context needed */
void rt_destroy(rt_ctx* ctx);
const char* rt_last_error(const rt_ctx* ctx);

/* Flatten-once upload: validates and copies the description, bakes the instance
 * transforms, builds the SAH BVH on the host, converts to the device layout and
 * uploads.  Replaces main.cpp:442 (bvh_node construction). */
int rt_upload_scene(rt_ctx* ctx, const rt_scene_desc* scene);

/* Animation update: replaces the uploaded scene by `scene`, which must have the STRUCTURE of the scene last uploaded
 * to ctx, without a tree build.  The tree keeps its topology and leaf order and its boxes are recomputed on the GPU.
 * Structure: every count of rt_scene_desc; each mesh's n_triangles and each image's size; the device kind of every
 * world primitive and boundary (sphere, moving sphere -- a non-zero center_vec --, quad, triangle); the quads of the
 * next-event emitter list (a quad with an emissive material and a non-zero area), in their order; each medium's
 * boundary class (one sphere, a six-quad box, general).  Anything else may change: transforms, centres, radii, motion,
 * corners, mesh positions, indices and uvs (checked like an upload), materials, textures, texels, Perlin tables, point
 * lights, media densities and the camera.
 * Every device record and table then equals the one rt_upload_scene(ctx, scene) would make, so frames equal a fresh
 * upload's bit for bit except for rays that hit two primitives at exactly the same t and, on a host-built scene with
 * several emitters, RT_FLAG_NEE (the emitter list keeps the uploaded tree's leaf order).  A refitted tree loosens as
 * objects move away from where it was built: upload again when render time grows (DESIGN.md section 10c).
 * RT_ERR_STATE without a scene, RT_ERR_INVALID for an invalid description or another structure (the message names
 * the first difference), RT_ERR_UNSUPPORTED when the scene is traversed as a wide tree (rt_set_bvh_width 4 / 8).
 * A refused refit changes nothing.  A refit waits for the passes in flight and treats the frame like rt_upload_scene:
 * a single-device context keeps its frame, moments and bound buffer; a multi-device context needs an rt_render before
 * its next download.  bvh_nodes, bvh_depth and bvh_leaves are unchanged; upload_ms and
 * upload_bytes report the refit.  An rt_upload_scene of the last uploaded scene afterwards may still reuse its staged
 * arena (scene_reused). */
int rt_refit_scene(rt_ctx* ctx, const rt_scene_desc* scene);

/* Which builder rt_upload_scene uses (replaces bvh.h:13-45 either way).
 *   1 host:   transforms baked, binned-SAH BVH2 and device records built on the CPU (best tree)
 *   2 device: raw arrays copied as they are; LBVH (Morton sort + radix tree) and device records
 *             built by CUDA kernels; subtrees of <= 128 primitives rebuilt with SAH (one warp each)
 *             and the top levels rebuilt with SAH on the host over a few thousand clusters:
 *             ~40x faster upload for million-primitive scenes, tree within a few % of the host's
 *   3 device, without the SAH top levels (pure LBVH; for comparison)
 *   0 auto:   device from 2^16 primitives up (environment RT_B200_BVH=host|device|lbvh overrides at rt_create)
 * Images do not depend on the choice (same records bit for bit, closest hit is tree-independent)
 * except where two primitives are hit at exactly the same t. */
int rt_set_bvh_builder(rt_ctx* ctx, int32_t mode);

/* Which acceleration structure the next rt_upload_scene builds for the render kernels (replaces
 * bvh.h:64-72 + aabb.h:61-85 either way): 2 = the SAH binary tree (64-byte nodes, two child boxes
 * each); 8 or 4 = the same tree collapsed into a wide BVH with 8-bit quantised child boxes and
 * octant-ordered child slots (csrc/bvh_wide.h).  Closest hits, and therefore images, do not depend on
 * the choice except where two primitives are hit at exactly the same t.  Scenes built by the device
 * builder keep the binary tree.  Environment RT_B200_BVH_WIDTH=2|4|8 sets the default at rt_create. */
int rt_set_bvh_width(rt_ctx* ctx, int32_t width);

/* Runs the whole bounce loop (Camera.txt:65-93, 177-272) for this context's
 * shard of samples [spp_begin, spp_begin + samples_per_pixel) and adds the
 * radiance into the accumulation buffer on the device.  Blocking unless
 * RT_FLAG_ASYNC. */
int rt_render(rt_ctx* ctx, const rt_render_params* params);
int rt_sync(rt_ctx* ctx);
/* Stream-ordered join, no host wait: whatever is enqueued on `stream` (a cudaStream_t of the context's device; NULL = the
 * context's own stream) after this call runs after every rt_render pass still in flight, RT_FLAG_OVERLAP passes included.
 * Single-device contexts take any stream; a multi-device context joins each device's passes into that device's own
 * stream (stream must be NULL). */
int rt_join(rt_ctx* ctx, void* stream);

/* Copy the finished frame to the host.  Either pointer may be NULL.
 *   rgb_linear: width*height*3 floats, radiance averaged over the accumulated spp,
 *               row-major top-down
 *   rgb8      : width*height*3 bytes, sqrt gamma, clamp [0,0.999], int(255.999*x)
 *               exactly as Camera.txt:77-89 (the buffer the reference hands to stbi_write_png)
 * `total_spp` is the divisor (pixel_samples_scale, Camera.txt:140): the number of
 * samples per pixel accumulated over all shards and passes. */
int rt_download(rt_ctx* ctx, int32_t total_spp, float* rgb_linear, uint8_t* rgb8);

/* Multi-view batches: n_views cameras of the uploaded scene rendered in one pass (one kernel launch), for turntables,
 * fly-throughs and multi-view datasets, without an rt_upload_scene per view.
 *
 * rt_render_views renders into a views frame of the context (n_views x height x width, view-major, 32 B per pixel like
 * the sums of rt_render).  View v is bit-identical to rt_render of the scene uploaded with cameras[v] and the same params
 * and seed (seeds[v] when seeds != NULL).  cameras[v].background must equal the uploaded camera's (RT_ERR_INVALID
 * otherwise), as must n_views >= 1 and cameras != NULL.
 *   - flags: RT_FLAG_ACCUMULATE, RT_FLAG_ASYNC, RT_FLAG_NEE and RT_FLAG_SHADOWED_POINT_LIGHTS; params->stream is honoured.
 *     RT_FLAG_STATS, RT_FLAG_MOMENTS, RT_FLAG_AOV, RT_FLAG_CAMERA_RAYS, RT_FLAG_COMPACT_TILES, RT_FLAG_OVERLAP, shard_count > 1 and multi-device contexts are
 *     RT_ERR_UNSUPPORTED, and so is a frame of n_views x width x height >= 2^31 slots.
 *   - the views frame is a buffer of its own: a views render does not touch the frame, moments or bound buffer of
 *     rt_render, and rt_render does not touch the views frame.
 *   - an RT_FLAG_ACCUMULATE pass must continue a views frame of the same (n_views, width, height), cameras and seeds
 *     (RT_ERR_STATE otherwise).
 *   - rt_stats: samples = n_views * width * height * samples_per_pixel, kernel_launches = 1, render_ms as for rt_render.
 * rt_download_views copies views [first, first + count) of the views frame to the host: count * height * width * 3 floats
 * / bytes, each view laid out like rt_download's planes.  Either pointer may be NULL.  RT_ERR_STATE before any views
 * render, RT_ERR_INVALID for a range outside the frame. */
int rt_render_views(rt_ctx* ctx, const rt_render_params* params,
                    const rt_camera* cameras, const uint64_t* seeds, int32_t n_views);
int rt_download_views(rt_ctx* ctx, int32_t total_spp, int32_t first, int32_t count,
                      float* rgb_linear, uint8_t* rgb8);

/* Deterministic primary-hit AOV for parity tests: casts the pixel-centre ray
 * ray(center, pixel00 + i*du + j*dv - center, time 0) over (0.001, inf) through
 * the same traversal/intersection code as rt_render, which decides WHICH primitive
 * is hit; t, point, normal and uv of that hit are then evaluated in double from the
 * double-precision ray (the reference's own formulas: sphere.h:33-58, quad.h:30-47,
 * triangle.h:67-110) and rounded to float once, so they can be held to 1e-5 against
 * the reference.  rt_probe_hit reports the FP32 completion the render kernels use.
 * Media are skipped (stochastic).  prim_id = -1 on a miss, otherwise the canonical primitive id
 * (rt_prim_ref: a mesh ref covers n_triangles consecutive ids).  Any output may be NULL. */
int rt_render_aov(rt_ctx* ctx, int32_t width, int32_t height,
                  int32_t* prim_id, float* t, float* normal /* 3 per pixel */,
                  float* point /* 3 per pixel */, float* uv /* 2 per pixel */);

/* The accumulation buffer: width*height*4 uint64 (R,G,B sums in 2^-RT_ACCUM_FRAC_BITS
 * fixed point, then the count of non-finite samples dropped).  Integer sums are
 * associative, so shards and progressive passes can be added in any order and the
 * frame stays bit-identical to the unsharded render.  rt_accum_buffer exposes
 * the device pointer (valid until the next rt_render with a different frame size,
 * rt_bind_accum or rt_destroy) so the caller can reduce it across GPUs with NCCL
 * (int64 SUM); rt_bind_accum makes the context render into a caller-owned device
 * buffer (e.g. a torch tensor) instead; NULL unbinds.  Both are for single-device contexts and full
 * (not compact) frames. */
#define RT_ACCUM_FRAC_BITS 28
int rt_accum_buffer(rt_ctx* ctx, void** device_ptr, size_t* bytes);
int rt_bind_accum(rt_ctx* ctx, void* device_ptr, size_t bytes, int32_t width, int32_t height);

/* Checkpoint / resume (replaces nothing in the reference, which restarts from scratch:
 * Camera.txt:65-93 keeps its sums in a local `color` per pixel).  rt_accum_download copies the
 * raw accumulation buffer (width*height*4 uint64) to the host; rt_accum_upload allocates a
 * width x height frame if needed and restores it.  Rendering on with RT_FLAG_ACCUMULATE and
 * spp_begin = the number of samples already in the buffer gives a frame bit-identical to an
 * uninterrupted render of the same total. */
int rt_accum_download(rt_ctx* ctx, uint64_t* host, size_t bytes);
int rt_accum_upload(rt_ctx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height);

/* Per-pixel noise of a frame rendered with RT_FLAG_MOMENTS.  A sample's value x in channel c is the integer its
 * radiance word adds (2^-28 units, clamped to [0, 2^20]); the moments hold S2 = sum x^2 exactly as two 48-bit limbs,
 * m[6p + 2c] = sum (x^2 mod 2^48), m[6p + 2c + 1] = sum (x^2 >> 48).  Like the sums they are bit-identical for any
 * device count, shard mode, pass split, overlap or resume.  A frame without valid moments is RT_ERR_STATE. */
/* Unbiased per-sample variance of every pixel and channel, s^2 = (n*S2 - S1^2) / (n*(n-1)) * 2^-56 with n = total_spp
 * (the rt_download divisor; dropped non-finite samples count as 0, as in the mean).  width*height*3 floats, row-major,
 * like rgb_linear: the same quantity as the `var` of the golden fixtures.  total_spp >= 2.  n*S2 - S1^2 is exact;
 * n*S2 saturates at 2^128 - 1, which only samples saturated at the 2^20 clamp at 65536 spp can reach.
 * Multi-device contexts: tile-sharded frames without a restored checkpoint (else RT_ERR_UNSUPPORTED). */
int rt_download_variance(rt_ctx* ctx, int32_t total_spp, float* variance);

/* Raw moments for checkpoints: width*height*6 uint64 (per channel: sum of the low and of the high 48 bits of x^2),
 * always the full frame like rt_accum_download.  rt_moments_upload restores the moments of the frame that
 * rt_accum_upload restored just before (RT_ERR_STATE otherwise).  Single-device contexts. */
int rt_moments_download(rt_ctx* ctx, uint64_t* host, size_t bytes);
int rt_moments_upload(rt_ctx* ctx, const uint64_t* host, size_t bytes, int32_t width, int32_t height);

/* Frame noise: the mean linear radiance over pixels and channels, and the RMS over pixels and channels of the
 * standard error of the pixel mean, sqrt(mean(s^2 / n)).  Reduced on the device as exact integer sums, so the result is
 * a pure function of the sums and moments: sum S1, and sum q with q = round(s^2 / n * 2^32) in double arithmetic
 * (saturating at 2^64 - 1), then divided once on the host.  Covers the pixels the context holds (a compact shard: its
 * own tiles).  Multi-device contexts: as rt_download_variance. */
int rt_frame_noise(rt_ctx* ctx, int32_t total_spp, double* mean_radiance, double* rms_std_error);

/* Auxiliary outputs of a frame rendered with RT_FLAG_AOV: the standard inputs of an external denoiser (albedo, normal)
 * and the depth of compositing, antialiased like the radiance because they come from the same camera samples.  They are
 * taken at the first event of each camera sample, with values the path computes there and no random number of its own:
 *   surface that scatters   albedo = the attenuation of the bounce (texture value for lambertian and isotropic, albedo for
 *                           metal -- also a sample the metal absorbs -- and specular, 1 for dielectric); normal = the
 *                           shading normal facing the ray (world space); depth = t |d|, the distance from the camera
 *                           ray's origin (on the lens when defocused); a hit
 *   light                   albedo = the emitted radiance clamped to [0, 1]; normal and depth as above; a hit
 *   medium scatter event    albedo = the isotropic attenuation; normal 0; depth = the distance to the event; a hit
 *   miss                    albedo = the background (rt_set_environment: the environment) clamped to [0, 1]; normal 0;
 *                           no depth; no hit
 * The sums are 8 uint64 per pixel: albedo x3 and depth unsigned, clamped to [0, 2^20], normal x3 signed (two's
 * complement), clamped to [-1, 1], all in 2^-RT_ACCUM_FRAC_BITS units, then the hit count.  A sample adds at most 2^48 to a
 * word (2^28 in magnitude to a normal word), so with at most 65536 samples per pixel no word overflows however the
 * samples are split -- save for 65536 samples all saturated at 2^20, the edge the radiance words share -- and, like the
 * radiance sums, they are bit-identical for any device count, shard, pass split, overlap or resume.
 * rt_download_aov writes width*height*8 floats, row-major and full-frame like rgb_linear (a compact shard: its own tiles,
 * zero elsewhere); per pixel albedo r, g, b, normal x, y, z, depth, coverage, each computed in double and rounded once to
 * float: albedo and normal sum / (2^28 n) with n = total_spp, depth sum / (2^28 hits) (0 without a hit), coverage hits / n.
 * So the albedo and the normal average over all n samples, misses included, and the depth over the samples that hit.
 * total_spp <= 0 is RT_ERR_INVALID, a frame without valid AOV sums RT_ERR_STATE.  Multi-device contexts: tile-sharded
 * frames without a restored checkpoint (else RT_ERR_UNSUPPORTED).  Ordered after outstanding hand-outs like rt_download. */
int rt_download_aov(rt_ctx* ctx, int32_t total_spp, float* aov);

/* Caller-defined cameras: one primary ray record per pixel, for camera models the uploaded pinhole cannot express
 * (fisheye and calibrated lenses, 360-degree panoramas, stereo rigs, the rays of a dataset).  A record holds the ray's
 * origin, its direction through the pixel centre (any non-zero length, like the rays of Camera.txt) and the change of
 * that direction per pixel in x and in y: the footprint the antialiasing jitter spans. */
typedef struct rt_camera_ray {
    float origin[3];
    float direction[3];
    float dx[3], dy[3];
} rt_camera_ray; /* 48 bytes; rt_struct_size(16) */

/* rt_set_camera_rays copies width*height records (row-major, top-down: rays[j*width + i] is pixel (i, j)) from host
 * memory into a buffer the context owns on each of its devices; the caller may free its copy when the call returns.
 * It waits for the passes in flight first.  rays == NULL frees the buffer.  RT_ERR_INVALID for width or height <= 0,
 * width*height >= 2^31, or a record with a non-finite value or a zero direction (the message names the first); a
 * refused call changes nothing.  rt_upload_scene and rt_refit_scene leave the rays as they are.
 * With RT_FLAG_CAMERA_RAYS, sample s of pixel (i, j) draws the camera uniforms u of Camera.txt:177-200 as rt_render does
 * and traces origin, direction + (u.x - 0.5) dx + (u.y - 0.5) dy (two FMAs per component, dy first) at time u.z, with no
 * defocus; a miss sees the uploaded camera's background.  Everything after the primary ray is unchanged, so a frame
 * rendered from the pinhole rays of the uploaded camera (origin = lookfrom, direction = pixel00 + i du + j dv - lookfrom,
 * dx = du, dy = dv) has the expectation of rt_render's, though not its bits.  The frame is the ordinary frame: every
 * download, checkpoint, shard and AOV call takes it as it is.
 * A frame accumulates passes of one source: the uploaded camera, or one rt_set_camera_rays call.  An RT_FLAG_ACCUMULATE
 * pass of the other source, or a rays pass after the rays were set again, is RT_ERR_STATE.  A frame restored with
 * rt_accum_upload (or bound with rt_bind_accum) accepts either, which is how a checkpointed rays render resumes. */
int rt_set_camera_rays(rt_ctx* ctx, const rt_camera_ray* rays, int32_t width, int32_t height);

/* Environment lighting: an equirectangular map of linear radiance that every ray leaving the scene sees, instead of the
 * camera's constant background -- image-based lighting, sky backgrounds, random HDRIs for synthetic data.
 * The map frame has +y up, -z at the image centre and +x to the right (camera::panorama_rays with lookfrom 0, lookat
 * (0, 0, -1) and vup +y, so pixel (i, j) of a width x height panorama looks at the centre of texel (i, j)).  rgb holds
 * width*height*3 floats, row-major, row 0 at the +y pole; rotation takes map directions to world directions (row-major). */
typedef struct rt_environment {
    const float* rgb;
    int32_t width, height;
    double rotation[9];
} rt_environment; /* rt_struct_size(17) */

/* rt_set_environment copies the map to every device of the context (the caller may free its texels when the call
 * returns), after the passes in flight, overlapped ones included.  env == NULL goes back to the camera's background.
 * RT_ERR_INVALID for rgb == NULL, width or height < 1, width*height >= 2^31, a texel that is negative or not finite, or a
 * rotation that is not orthonormal with determinant +1 within 1e-6 (the message names the first); a refused call changes
 * nothing.  rt_upload_scene and rt_refit_scene keep the environment, and setting it does not touch the frame.
 * The radiance of a ray with direction d that leaves the scene (in FP32):
 *   1. m = R^T d, R = rotation
 *   2. phi = atan2(m.x, -m.z), theta = atan2(m.y, sqrt(m.x^2 + m.z^2))
 *   3. tx = (phi / (2 pi) + 1/2) width - 1/2, ty = (1/2 - theta / pi) height - 1/2
 *   4. bilinear between texels floor(tx), floor(tx) + 1 (columns modulo width) and floor(ty), floor(ty) + 1 (rows
 *      clamped to [0, height - 1]), each lerp a + t (b - a), so that a uniform map returns its texel exactly: a map of
 *      texels equal to the background renders the frame of the background bit for bit.
 * While an environment is set it replaces the background in every render: rt_render with any flags, shards, compact
 * tiles, overlapped passes and multi-device contexts, and rt_render_views (whose rule on cameras[v].background stays).
 * With RT_FLAG_AOV a miss reports the environment clamped to [0, 1] as its albedo.  With RT_FLAG_NEE the environment is
 * gathered only by the paths whose BSDF-sampled direction leaves the scene, at full weight: NEE samples the listed quad
 * emitters only, so no other technique covers those directions and the estimate stays unbiased.  RT_FLAG_STATS is
 * RT_ERR_UNSUPPORTED while an environment is set, and a wide tree (rt_set_bvh_width) is traversed as the binary tree. */
int rt_set_environment(rt_ctx* ctx, const rt_environment* env);

/* Compact tile buffers across processes (one process per GPU, e.g. under torchrun; single-device contexts):
 *   rt_shard_pixels   slots of the compact buffer of shard (rank, count): its tiles x tile_size^2 (edge tiles padded)
 *   rt_resolve_tiles  the compact sums of the last RT_FLAG_COMPACT_TILES render -> averaged radiance (3 floats per slot)
 *                     and / or RGB8 (3 bytes per slot, Camera.txt:77-89) in CALLER-OWNED DEVICE buffers of
 *                     capacity_pixels slots each, ready for an NCCL gather by the caller
 *   rt_untile         `shard_count` such buffers side by side on this context's device (shard r at
 *                     dev_shards + r * shard_stride_bytes) -> the full row-major frame in host memory;
 *                     bytes_per_pixel 3 (RGB8), 12 (float RGB) or 32 (raw sums) */
size_t rt_shard_pixels(int32_t width, int32_t height, int32_t tile_size, int32_t shard_rank, int32_t shard_count);
int rt_resolve_tiles(rt_ctx* ctx, int32_t total_spp, float* dev_rgb_linear, uint8_t* dev_rgb8, size_t capacity_pixels);
int rt_untile(rt_ctx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count,
              int32_t width, int32_t height, int32_t tile_size, void* host_out);

/* Asynchronous hand-out of the frame: the copy to host memory overlaps the next pass.
 *   rt_download_begin  like rt_download, but returns once the resolve and the device-to-host copy are QUEUED (the
 *                      copy on a stream of its own, into pinned host memory owned by the context); the next
 *                      rt_upload_scene / rt_render may be issued at once
 *   rt_untile_begin    like rt_untile (bytes_per_pixel 3 or 12), same hand-out
 *   rt_frame_end       waits for the OLDEST outstanding begin and returns pointers into the context's pinned
 *                      buffer (NULL for a plane that was not asked for), valid until two more begins; at most two
 *                      frames may be outstanding
 * Synchronous readbacks (rt_download, rt_download_variance, rt_accum_download, ...) issued while a frame is outstanding
 * are ordered after its copy, so rt_frame_end returns the frame as it was at its begin. */
int rt_download_begin(rt_ctx* ctx, int32_t total_spp, int32_t want_linear, int32_t want_rgb8);
int rt_untile_begin(rt_ctx* ctx, const void* dev_shards, size_t shard_stride_bytes, int32_t bytes_per_pixel, int32_t shard_count,
                    int32_t width, int32_t height, int32_t tile_size);
int rt_frame_end(rt_ctx* ctx, const float** rgb_linear, const uint8_t** rgb8);

int rt_get_stats(rt_ctx* ctx, rt_stats* out);

/* sizeof() of the ABI structs as this library was compiled, so that a foreign-language
 * binding (ctypes, cgo, JNI ...) can verify its own declarations at load time.
 * which: 0 rt_scene_desc, 1 rt_render_params, 2 rt_stats, 3 rt_sphere, 4 rt_quad,
 * 5 rt_triangle, 6 rt_medium, 7 rt_material, 8 rt_texture, 9 rt_image, 10 rt_perlin,
 * 11 rt_point_light, 12 rt_camera, 13 rt_xform, 14 rt_prim_ref, 15 rt_mesh, 16 rt_camera_ray, 17 rt_environment;
 * 0 for anything else. */
size_t rt_struct_size(int which);

/* FP32 FMA issue-rate microbenchmark on the context's device, for the FP32
 * roofline denominator (not in MEASURED_PEAKS.json).  Returns TFLOP/s. */
int rt_measure_fp32_peak(rt_ctx* ctx, double* tflops);
/* L1 load-bandwidth microbenchmark (128-bit loads over an L1-resident window per block), GB/s: the denominator
 * of the node/primitive-bytes figure -- the BASELINE scenes are cache-resident, their bytes are not HBM bytes. */
int rt_measure_l1_peak(rt_ctx* ctx, double* gbs);

/* Per-function device probes for known-answer tests: evaluate one hot-path
 * function on the device for n inputs (host pointers).  `texture` / `material` are indices into the uploaded
 * tables; an index outside them is RT_ERR_INVALID.
 *   rt_probe_texture: texture::value (texture.h) for n (u,v,p) tuples.
 *   rt_probe_scatter: material::emitted + material::scatter (material.h) with the
 *     four uniforms the bounce would have drawn supplied by the caller:
 *     u[0..2] feed random_unit_vector (vec3.h:107-115), u[3] the dielectric test.
 *   rt_probe_hit: closest hit of arbitrary rays (origin, direction, time, t_min,
 *     t_max) against the uploaded world, media skipped. */
int rt_probe_texture(rt_ctx* ctx, int32_t texture, int32_t n,
                     const float* uvp /* n*5: u v px py pz */, float* rgb /* n*3 */);
int rt_probe_scatter(rt_ctx* ctx, int32_t material, int32_t n,
                     const float* in /* n*16: o[3] d[3] time p[3] normal[3] front u v */,
                     const float* uniforms /* n*4 */,
                     float* out /* n*16 floats, 64 bytes per record: [0] scattered (1/0), [1..3] attenuation,
                                   [4..6] scattered origin, [7..9] scattered direction, [10..12] emitted,
                                   [13] scattered time, [14..15] zero */);
int rt_probe_hit(rt_ctx* ctx, int32_t n, const float* rays /* n*9: o[3] d[3] time tmin tmax */,
                 int32_t* prim_id, float* t, float* normal, float* uv);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
