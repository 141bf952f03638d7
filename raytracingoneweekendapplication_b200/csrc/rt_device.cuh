// rt_device.cuh — device-side data layout and the hot-path functions of the path tracer
// (sm_100a).  Everything here is FP32 unless a function says otherwise.
//
// Layout in HBM (all read-only during a render, fetched through the non-coherent path,
// L1/L2 resident for every BASELINE scene; see DESIGN.md "data layout"):
//   nodes      interior BVH2 nodes, 64 B = 4 x float4:
//                {L.min, link_L} {L.max, link_R} {R.min, -} {R.max, -}
//              link >= 0: interior node index; link < 0: leaf, ~link =
//                type<<28 | (count-1)<<25 | first     (first indexes the typed array)
//   sph        static spheres, 16 B  {c.xyz, r}
//   msph       moving spheres, 32 B  {c0.xyz, r} {cvec.xyz, 0}
//   quad       48 B  {n.xyz, D} {A.xyz, a0} {B.xyz, b0}   alpha = A.P - a0, beta = B.P - b0
//   tri        48 B  {p0.xyz, 0} {e1.xyz, 0} {e2.xyz, 0}
//   *_d        FP64 copies: sphere paths of the render kernels (near-surface roots, refinement of the
//              accepted hit) and complete_hit_fp64 of the deterministic rays (AOV, probes)
//   *_sh       shading records fetched once per accepted hit
// Typed arrays are stored in BVH leaf order, so a leaf's primitives are contiguous and
// there is no index indirection.  Media boundaries live at the tail of the same arrays.
#pragma once
#include <cuda_runtime.h>

#include <stddef.h>
#include <stdint.h>
#include "rt_b200.h"

namespace rtdev {

enum : uint32_t { PT_SPHERE = 0, PT_MSPHERE = 1, PT_QUAD = 2, PT_TRI = 3 };
constexpr uint32_t PRIM_NONE = 0xffffffffu;
constexpr int STACK_SIZE = 64;  // levels a tree may have (checked at upload); BVH2 depth of a SAH tree over 2^25 prims stays below

struct DevMaterial {  // 32 B
    int type;
    int tex;
    float albedo[3];
    float param;
    int needs_uv;  // the texture chain reads (u,v): sphere UVs are only computed then
    int pad;
};
struct DevTexture {  // 32 B
    int type;
    int a;  // checker: even, image: image index, noise: perlin index
    int b;  // checker: odd
    float scale;
    float color[3];
    int pad;
};
struct DevImage {
    const unsigned char* rgb;
    int w, h;
};
struct DevMedium {  // 48 B
    int bfirst, bcount;  // range in `boundary`
    float neg_inv_density;  // -1 / (multiplicity * density)
    int material;
    float normal[3];  // R * (1,0,0)
    int sphere;  // >= 0: the boundary is this one static sphere (index into sph); -1: generic
    int box;     // >= 0: the boundary is the six quads of one box() (any rigid transform): three slabs, media_box + 4 * box
    int pad[3];
};
// A quad emitter the opt-in next-event estimation samples (SURVEY 8f rank 4): world-space
// corner and edges, area, emission texture, and the running share of the total emitter area.
struct DevNeeLight {  // 64 B
    float Q[3];
    float area;
    float u[3];
    int tex;
    float v[3];
    float cdf;  // sum of the areas up to and including this light / total area
    float n[3];
    int pad;
};
struct DevLight {
    float pos[3];
    float size;
    float intensity[3];
    float pad;
};

struct DevScene {
    const float4* nodes;
    int root;
    int n_nodes;
    int n_world;  // 0: every ray misses (the root link is not followed)
    uint32_t env_lo;  // the environment map of rt_set_environment (env_radiance), its two 32-bit halves in two alignment
                      // holes (here and after n_media), so that no field or kernel parameter offset moves; only the ENV
                      // instances read them.  Stamped on the launch's copy of the scene (launch_v2)
    // the W-wide quantised BVH collapsed from `nodes` (bvh_wide.h; null when the scene has none):
    // W = 8: 5 uint4 per node, W = 4: 3; wrefs[W * node + slot] = BVH2 leaf link of a leaf child
    const void* wnodes;
    const int32_t* wrefs;
    int wide_width;  // 0, 4 or 8
    uint32_t f32_one_bits;  // 0x3F800000, as a kernel parameter the compiler cannot fold (rt_wide.cuh, unit_plus_byte)
    const float4* sph;
    const float4* msph;
    const float4* quad;
    const float4* tri;
    const double* sph_d;   // 4 per sphere: c, r
    const double* msph_d;  // 8 per sphere: c0, r, cvec, 0
    const double* quad_d;  // 12 per quad: n, D, A, a0, B, b0
    const double* tri_d;   // 9 per triangle: p0, e1, e2
    const int4* sph_sh;    // {material, xform, prim id, 0}
    const int4* msph_sh;
    const int4* quad_sh;   // {material, 0, prim id, 0}
    const float4* tri_sh;  // 3 per triangle: {n.xyz, as_float(material)} {uv0, uv1} {uv2, as_float(id), 0}
    const float* xrot;     // 9 per xform: world-from-object rotation, row-major
    const DevMedium* media;
    const float4* media_box;  // per box-bounded medium: {axis0, lo0} {axis1, lo1} {axis2, lo2} {hi0, hi1, hi2, -}
    int n_media;
    uint32_t env_hi;
    const uint32_t* boundary;  // packed prim refs type<<28 | index
    const DevMaterial* mats;
    const DevTexture* texs;
    const DevImage* images;
    const float4* perlin_vec;          // 256 per perlin
    const unsigned char* perlin_perm;  // 768 per perlin: perm_x, perm_y, perm_z
    const DevLight* lights;
    int n_lights;
    const DevNeeLight* nee_lights;  // RT_FLAG_NEE: quads with an emissive material
    int n_nee_lights;
    float nee_total_area;
    // camera (Camera.txt:136-175, evaluated in double on the host)
    float center[3], dir00[3], du[3], dv[3], disk_u[3], disk_v[3];
    float background[3];
    int defocus;
    __host__ __device__ const float4* env() const { return (const float4*)(((uint64_t)env_hi << 32) | env_lo); }
    void set_env(const void* p) { env_lo = (uint32_t)(uintptr_t)p; env_hi = (uint32_t)((uint64_t)(uintptr_t)p >> 32); }
};
static_assert(sizeof(DevScene) == 344 && offsetof(DevScene, env_lo) == 20 && offsetof(DevScene, wnodes) == 24 &&
                  offsetof(DevScene, env_hi) == 172 && offsetof(DevScene, boundary) == 176,
              "the environment pointer fills alignment holes only");

// One camera of a multi-view batch (rt_render_views): the camera block of DevScene for that view's camera and frame,
// and the Philox key of its seed.  96 B.
struct ViewRecord {
    float center[3], dir00[3], du[3], dv[3], disk_u[3], disk_v[3];
    int defocus;
    uint32_t k0, k1;
    uint32_t pad[3];
};

struct Stats {
    unsigned long long rays, node_visits, box_tests, sphere_tests, quad_tests, tri_tests, medium_queries,
        boundary_tests, fp64_sphere, nonfinite, samples;
    // lane occupancy of render_kernel_v2's phases, counted per warp-level iteration (lane 0 adds)
    unsigned long long desc_iters, desc_lanes, desc_trav_lanes, leaf_iters, leaf_lanes, shade_iters, shade_lanes;
    unsigned long long empty_steps;  // node steps in which no child box was hit
};

// ---------------------------------------------------------------------------------
// small vector helpers
// ---------------------------------------------------------------------------------
struct V3 {
    float x, y, z;
};
__device__ __forceinline__ V3 v3(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 v3(const float* p) { return V3{p[0], p[1], p[2]}; }
__device__ __forceinline__ V3 v3(float4 f) { return V3{f.x, f.y, f.z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator-(V3 a) { return V3{-a.x, -a.y, -a.z}; }
__device__ __forceinline__ V3 operator*(V3 a, V3 b) { return V3{a.x * b.x, a.y * b.y, a.z * b.z}; }
__device__ __forceinline__ V3 operator*(float s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return V3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ float dot(V3 a, V3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
__device__ __forceinline__ V3 cross(V3 a, V3 b) {
    return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ V3 fma3(float s, V3 a, V3 b) { return V3{fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)}; }
__device__ __forceinline__ V3 normalize(V3 a) { return rsqrtf(dot(a, a)) * a; }

__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }

// a * s + t on both halves in one instruction (FFMA2, new with sm_100; the scalars are broadcast operands)
__device__ __forceinline__ float2 ffma2(float2 a, float s, float t) {
    unsigned long long ra = (unsigned long long)__float_as_uint(a.x) | ((unsigned long long)__float_as_uint(a.y) << 32);
    unsigned long long rs = (unsigned long long)__float_as_uint(s) | ((unsigned long long)__float_as_uint(s) << 32);
    unsigned long long rt = (unsigned long long)__float_as_uint(t) | ((unsigned long long)__float_as_uint(t) << 32);
    unsigned long long rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rs), "l"(rt));
    return make_float2(__uint_as_float((unsigned)rd), __uint_as_float((unsigned)(rd >> 32)));
}

// ---------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter = (pixel, sample, bounce<<8 | stream, 0),
// key = seed.  The image is a pure function of these, which is what makes 1/2/4/8-GPU
// renders bit-identical.  Dimension assignment (shared with oracle/philox_ref.h):
//   stream 0        camera: x = jitter x, y = jitter y, z = ray time
//   stream 1..15    defocus-disk rejection attempts, two per block ((x,y) then (z,w))
//   stream 16       scatter: x,y,z = random_unit_vector's cube point, w = dielectric test
//   stream 32 + k   media 4k..4k+3: one free-flight uniform each
// ---------------------------------------------------------------------------------
constexpr uint32_t RS_CAMERA = 0, RS_DEFOCUS = 1, RS_SCATTER = 16, RS_NEE = 24, RS_MEDIUM = 32;

// inlined: out of line it costs 10 % on C5 (call ABI spills)
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// 24-bit uniform in [0,1): exactly representable in FP32 and identical in the FP64 oracle
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }

struct Rng {
    uint32_t pixel, sample, k0, k1;
    __device__ __forceinline__ float4 draw(uint32_t bounce, uint32_t stream) const {
        uint4 r = philox4x32_10(pixel, sample, (bounce << 8) | stream, 0u, k0, k1);
        return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
    }
};

// ---------------------------------------------------------------------------------
// ray + hit
// ---------------------------------------------------------------------------------
struct Ray {
    V3 o, d;
    float time;
};
struct Hit {
    float t;
    uint32_t prim;  // type<<28 | index, PRIM_NONE = miss
    float u, v;     // quad: alpha, beta; triangle: barycentric u, v
};

// sphere.h:33-46 verbatim in double.  Out of line: it is the rare path (a ray that starts within
// r/16 of the surface of a sphere it did not start on) and keeping its DFMA/DSQRT/DDIV
// sequences out of the traversal loop shrinks the loop's code and register footprint.
// Returns the two roots, or NaN for both when the line misses the sphere: every caller rejects a NaN root with
// the same interval test it applies to a real one.  The ray comes by value and the roots go back by value: an
// argument by reference would give the caller's ray and roots an address, and so a home in local memory.
__device__ __noinline__ float2 sphere_roots_fp64(const double* cd, bool moving, Ray ray) {
    double cx = cd[0], cy = cd[1], cz = cd[2], rr = cd[3];
    if (moving) {
        cx += (double)ray.time * cd[4]; cy += (double)ray.time * cd[5]; cz += (double)ray.time * cd[6];
    }
    double ox = cx - (double)ray.o.x, oy = cy - (double)ray.o.y, oz = cz - (double)ray.o.z;
    double dx = ray.d.x, dy = ray.d.y, dz = ray.d.z;
    double a = dx * dx + dy * dy + dz * dz;
    double hh = dx * ox + dy * oy + dz * oz;
    double cc = ox * ox + oy * oy + oz * oz - rr * rr;
    double disc = hh * hh - a * cc;
    if (disc < 0.0) return make_float2(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff));
    double sq = sqrt(disc);
    return make_float2((float)((hh - sq) / a), (float)((hh + sq) / a));
}

// sphere.h:32-49.  Robust FP32 form (distance from the centre to the ray line instead of
// h*h - a*c), the exact c = 0 case for a ray that starts ON this sphere, and the
// reference's own double-precision quadratic when the origin is within r/16 of the
// surface of a sphere it did not start on (large ground spheres).
template <bool STATS>
__device__ __forceinline__ void hit_sphere(V3 c, float r, const double* cd, bool moving, bool self, const Ray& ray, float inv_a,
                                           float tmin, uint32_t prim, Hit& hit, Stats* st) {
    V3 oc = c - ray.o;
    float h = dot(ray.d, oc);
    float k = h * inv_a;
    float r2 = r * r;
    float t0, t1;
    if (self) {
        t0 = -1.0f;  // the root at the origin (exactly 0 in the reference up to 1e-13)
        t1 = 2.0f * k;
    } else {
        float cterm = dot(oc, oc) - r2;
        if (fabsf(cterm) < 0.125f * r2) {
            if (STATS) st->fp64_sphere++;
            const float2 roots = sphere_roots_fp64(cd, moving, ray);  // NaN: no root passes the test below
            t0 = roots.x;
            t1 = roots.y;
        } else {
            V3 l = fma3(-k, ray.d, oc);
            float disc = r2 - dot(l, l);
            if (disc < 0.0f) return;
            float sq = sqrtf(disc * inv_a);
            t0 = k - sq;
            t1 = k + sq;
        }
    }
    float t = t0;
    if (!(t > tmin && t < hit.t)) {  // interval::surrounds (sphere.h:45-48)
        t = t1;
        if (!(t > tmin && t < hit.t)) return;
    }
    hit.t = t;
    hit.prim = prim;
}

// quad.h:29-73 with alpha = w.(p x v) rewritten as (v x w).p (A = v x w, B = w x u)
__device__ __forceinline__ void hit_quad(float4 q0, float4 q1, float4 q2, const Ray& ray, float tmin, uint32_t prim, Hit& hit) {
    V3 n = v3(q0);
    float denom = dot(n, ray.d);
    if (fabsf(denom) < 1e-8f) return;
    float t = __fdividef(q0.w - dot(n, ray.o), denom);
    if (!(t >= tmin && t <= hit.t)) return;  // interval::contains (quad.h:39)
    V3 p = fma3(t, ray.d, ray.o);
    float alpha = dot(v3(q1), p) - q1.w;
    float beta = dot(v3(q2), p) - q2.w;
    if (alpha < 0.0f || alpha > 1.0f || beta < 0.0f || beta > 1.0f) return;
    hit.t = t;
    hit.prim = prim;
    hit.u = alpha;
    hit.v = beta;
}

// triangle.h:65-113 (Moeller-Trumbore, two-sided, edges precomputed)
__device__ __forceinline__ void hit_tri(float4 t0, float4 t1, float4 t2, const Ray& ray, float tmin, uint32_t prim, Hit& hit) {
    V3 e1 = v3(t1), e2 = v3(t2);
    V3 pvec = cross(ray.d, e2);
    float det = dot(e1, pvec);
    if (fabsf(det) < 1e-8f) return;
    float inv = __fdividef(1.0f, det);
    V3 tvec = ray.o - v3(t0);
    float u = dot(tvec, pvec) * inv;
    if (u < 0.0f || u > 1.0f) return;
    V3 qvec = cross(tvec, e1);
    float v = dot(ray.d, qvec) * inv;
    if (v < 0.0f || u + v > 1.0f) return;
    float t = dot(e2, qvec) * inv;
    if (t < tmin || t > hit.t) return;
    hit.t = t;
    hit.prim = prim;
    hit.u = u;
    hit.v = v;
}

// LITE: the scene has no triangles (and, elsewhere, no point lights and no defocus): the
// production kernel is also compiled without those features, because in one megakernel every
// feature costs every scene registers and instruction-cache (C5 +4 % without them).
// MSPH = false: the scene has no moving sphere (instance without that code).
template <bool STATS, bool LITE = false, bool MSPH = true>
__device__ __forceinline__ void hit_prim(const DevScene& S, uint32_t type, uint32_t idx, const Ray& ray, float inv_a, float tmin,
                                         uint32_t origin_prim, Hit& hit, Stats* st) {
    uint32_t prim = (type << 28) | idx;
    if (MSPH ? type <= PT_MSPHERE : type == PT_SPHERE) {
        // static and moving spheres share ONE inlined copy of the test (and one call site of the FP64 roots): only the
        // fetch of the centre differs (sphere.h:33 center.at(r.time())) -- two copies cost C5, which has one moving
        // sphere, 4 % (round 2)
        if (STATS) st->sphere_tests++;
        float4 s;
        const double* cd;
        const bool moving = MSPH && type == PT_MSPHERE;
        if (!moving) {
            s = ldg4(S.sph + idx);
            cd = S.sph_d + 4 * (size_t)idx;
        } else {
            const float4* m = S.msph + 2 * (size_t)idx;
            const float4 a = ldg4(m), b = ldg4(m + 1);
            const V3 c = fma3(ray.time, v3(b), v3(a));
            s = make_float4(c.x, c.y, c.z, a.w);
            cd = S.msph_d + 8 * (size_t)idx;
        }
        hit_sphere<STATS>(v3(s), s.w, cd, moving, prim == origin_prim, ray, inv_a, tmin, prim, hit, st);
    } else if (type == PT_QUAD) {
        if (STATS) st->quad_tests++;
        if (prim == origin_prim) return;  // a ray leaving a planar primitive cannot hit it again
        const float4* q = S.quad + 3 * (size_t)idx;
        hit_quad(ldg4(q), ldg4(q + 1), ldg4(q + 2), ray, tmin, prim, hit);
    } else if (!LITE && type == PT_TRI) {
        if (STATS) st->tri_tests++;
        if (prim == origin_prim) return;
        const float4* t = S.tri + 3 * (size_t)idx;
        hit_tri(ldg4(t), ldg4(t + 1), ldg4(t + 2), ray, tmin, prim, hit);
    }
}

// bvh.h:64-72 + aabb.h:61-85 + hittable_list.h:22-35, as an iterative stack traversal of the
// flattened SAH tree: closest hit over (tmin, tmax).
//
// The traversal is a resumable state machine (Trav) so that the megakernel can suspend a
// lane's ray between steps: `interior()` consumes one 64-byte node (two child boxes), `leaf()`
// intersects the primitives of one leaf, both end by choosing the next link or popping the
// stack; `done()` turns true when the stack runs dry.
struct RayConst {  // per-ray constants of the slab test, recomputed when a traversal phase starts
    float idx, idy, idz, ox, oy, oz, inv_a;
    __device__ __forceinline__ void set(const Ray& ray) {
        // __frcp_rn: the correctly rounded reciprocal (same value as 1.0f / x) without the generic
        // division's slow path -- this runs for every lane at the start of every traversal phase
        auto safe_inv = [](float d) { return __frcp_rn(fabsf(d) > 1e-30f ? d : copysignf(1e-30f, d)); };
        idx = safe_inv(ray.d.x); idy = safe_inv(ray.d.y); idz = safe_inv(ray.d.z);
        ox = ray.o.x * idx; oy = ray.o.y * idy; oz = ray.o.z * idz;
        inv_a = __frcp_rn(dot(ray.d, ray.d));
    }
};

constexpr int LINK_DONE = (int)0x80000000;
  // negative, and not a leaf encoding (those are > -2^30)

// Traversal state.  The stack is a separate local array of packed (entry distance, link)
// pairs: keeping the scalars out of the indexed array lets the compiler hold them in
// registers, and one 64-bit local store/load moves an entry.
typedef unsigned long long StackEntry;
__device__ __forceinline__ StackEntry pack_entry(int link, float t) {
    return ((unsigned long long)__float_as_uint(t) << 32) | (unsigned)link;
}

struct Trav {
    Hit hit;
    int cur;  // >= 0 interior node, < 0 leaf, LINK_DONE finished (also < 0)
    int sp;

    __device__ __forceinline__ void init(const DevScene& S, float tmax) {
        hit.t = tmax;
        hit.prim = PRIM_NONE;
        hit.u = hit.v = 0.0f;
        sp = 0;
        cur = S.n_world > 0 ? S.root : LINK_DONE;
    }
    __device__ __forceinline__ bool done() const { return cur == LINK_DONE; }
    // the interface render_kernel_v2 shares with the wide traversal (rt_wide.cuh)
    __device__ __forceinline__ void clear() { cur = LINK_DONE; sp = 0; }
    __device__ __forceinline__ bool wants_node() const { return cur >= 0; }

    // pop, skipping subtrees that start beyond the closest hit so far
    __device__ __forceinline__ void pop(const StackEntry* stack) {
        cur = LINK_DONE;
        while (sp > 0) {
            sp--;
            const StackEntry e = stack[sp];
            if (__uint_as_float((unsigned)(e >> 32)) <= hit.t) {
                cur = (int)(unsigned)e;
                break;
            }
        }
    }

    // One 64-byte node = two child boxes (aabb.h:61-85 twice).  The choice of the next link is
    // select-based: the four outcomes (both / left / right / none) share one instruction stream,
    // the push is a predicated store, and only the (rare) "none" case branches into pop().
    template <bool STATS>
    __device__ __forceinline__ void interior(const DevScene& S, const RayConst& rc, float tmin, StackEntry* stack, Stats* st) {
        const float4* n = S.nodes + 4 * (size_t)cur;
        float4 a = ldg4(n), b = ldg4(n + 1), c = ldg4(n + 2), e = ldg4(n + 3);
        if (STATS) { st->node_visits++; st->box_tests += 2; }
        // paired layout (pair_nodes): the same plane of the left and the right box sit side by side, so one
        // FFMA2 (fma.rn.f32x2, sm_100) moves both to ray space -- 6 instructions instead of 12, same values
        const float2 x0 = ffma2(make_float2(a.x, a.y), rc.idx, -rc.ox), y0 = ffma2(make_float2(a.z, a.w), rc.idy, -rc.oy);
        const float2 z0 = ffma2(make_float2(b.x, b.y), rc.idz, -rc.oz), x1 = ffma2(make_float2(b.z, b.w), rc.idx, -rc.ox);
        const float2 y1 = ffma2(make_float2(c.x, c.y), rc.idy, -rc.oy), z1 = ffma2(make_float2(c.z, c.w), rc.idz, -rc.oz);
        const float lx0 = x0.x, rx0 = x0.y, ly0 = y0.x, ry0 = y0.y, lz0 = z0.x, rz0 = z0.y;
        const float lx1 = x1.x, rx1 = x1.y, ly1 = y1.x, ry1 = y1.y, lz1 = z1.x, rz1 = z1.y;
        const int linkl = __float_as_int(e.x), linkr = __float_as_int(e.y);
        float ln = fmaxf(fmaxf(fminf(lx0, lx1), fminf(ly0, ly1)), fmaxf(fminf(lz0, lz1), tmin));
        float lf = fminf(fminf(fmaxf(lx0, lx1), fmaxf(ly0, ly1)), fminf(fmaxf(lz0, lz1), hit.t));
        float rn = fmaxf(fmaxf(fminf(rx0, rx1), fminf(ry0, ry1)), fmaxf(fminf(rz0, rz1), tmin));
        float rf = fminf(fminf(fmaxf(rx0, rx1), fmaxf(ry0, ry1)), fminf(fmaxf(rz0, rz1), hit.t));
        const bool hl = ln <= lf, hr = rn <= rf;
        if (STATS && !hl && !hr) st->empty_steps++;
        const bool right_first = hr && (!hl || rn < ln);
        const int near_l = right_first ? linkr : linkl;
        const int far_l = right_first ? linkl : linkr;
        const float far_t = right_first ? ln : rn;
        if (hl && hr) {
            // no bounds check here: a ray's stack never holds more entries than the tree has levels, and
            // rt_upload_scene guarantees fewer than STACK_SIZE levels when the tree is uploaded -- it refuses
            // (host path) or rebuilds on the host (device path) a deeper tree.  A device-side check costs 2.5 % on C5.
            stack[sp] = pack_entry(far_l, far_t);
            sp++;
        }
        if (hl || hr) cur = near_l;
        else pop(stack);
    }

    template <bool STATS, bool LITE = false, bool MSPH = true>
    __device__ __forceinline__ void leaf(const DevScene& S, const Ray& ray, const RayConst& rc, float tmin, uint32_t origin_prim,
                                         StackEntry* stack, Stats* st) {
        uint32_t v = ~(uint32_t)cur;
        uint32_t type = v >> 28, cnt = ((v >> 25) & 7u) + 1u, first = v & 0x1ffffffu;
        for (uint32_t i = 0; i < cnt; i++) hit_prim<STATS, LITE, MSPH>(S, type, first + i, ray, rc.inv_a, tmin, origin_prim, hit, st);
        pop(stack);
    }

    template <bool STATS>
    __device__ __forceinline__ void node_step(const DevScene& S, const Ray&, const RayConst& rc, float tmin, StackEntry* stack, Stats* st) {
        interior<STATS>(S, rc, tmin, stack, st);
    }
    template <bool STATS, bool LITE, bool MSPH = true>
    __device__ __forceinline__ void leaf_step(const DevScene& S, const Ray& ray, const RayConst& rc, float tmin, uint32_t origin_prim,
                                              StackEntry* stack, Stats* st) {
        leaf<STATS, LITE, MSPH>(S, ray, rc, tmin, origin_prim, stack, st);
    }
};

__device__ __forceinline__ void traverse(const DevScene& S, const Ray& ray, float tmin, float tmax, uint32_t origin_prim, Hit& hit) {
    RayConst rc;
    rc.set(ray);
    Trav tr;
    StackEntry stack[STACK_SIZE];
    tr.init(S, tmax);
    StackEntry* const sp_ = stack;
    while (!tr.done()) {
        if (tr.cur >= 0) tr.interior<false>(S, rc, tmin, sp_, nullptr);
        else tr.leaf<false>(S, ray, rc, tmin, origin_prim, sp_, nullptr);
    }
    hit = tr.hit;
}

// The two boundary->hit calls of constant_medium.h:23-27 against an arbitrary boundary (no
// BVH: a boundary is one sphere or the six quads of a box in every scene of the reference).
// Out of line: only media whose boundary is not a single static sphere come here.  Returns (t1, t2), NaN for both
// when the line is no boundary pair; by value as in sphere_roots_fp64.
__device__ __noinline__ float2 boundary_pair_generic(const DevScene& S, int bfirst, int bcount, Ray ray, float inv_a) {
    const float inf = __int_as_float(0x7f800000), nan = __int_as_float(0x7fffffff);
    Hit h;
    h.t = inf; h.prim = PRIM_NONE; h.u = h.v = 0.0f;
    for (int i = 0; i < bcount; i++) {
        uint32_t ref = __ldg(S.boundary + bfirst + i);
        hit_prim<false>(S, ref >> 28, ref & 0x0fffffffu, ray, inv_a, -inf, PRIM_NONE, h, nullptr);  // interval::universe
    }
    if (h.prim == PRIM_NONE) return make_float2(nan, nan);
    const float t1 = h.t;
    h.t = inf; h.prim = PRIM_NONE;
    for (int i = 0; i < bcount; i++) {
        uint32_t ref = __ldg(S.boundary + bfirst + i);
        hit_prim<false>(S, ref >> 28, ref & 0x0fffffffu, ray, inv_a, t1 + 0.0001f, PRIM_NONE, h, nullptr);
    }
    if (h.prim == PRIM_NONE) return make_float2(nan, nan);
    return make_float2(t1, h.t);
}

// The same two calls against a boundary that is ONE box() (box() in quad.h: six quads, the faces of a parallelepiped;
// both smoke volumes of the Cornell scene): the line enters the closed box at the nearest of the (at most two) faces it
// crosses -- what hit(universe) over the six quads returns -- and leaves it at the other one -- what hit(t1 + 1e-4, inf)
// returns; both come out of ONE three-slab test instead of twelve quad tests.  A line that misses the box, or only
// touches it (exit within 1e-4 of the entry), is no boundary pair, as there.  quad.h:35's parallel-plane rejection
// (|n.d| < 1e-8) becomes the slab's inside/outside test for that axis.  Returns (t1, t2) as boundary_pair_generic does.
__device__ __noinline__ float2 boundary_pair_box(const float4* __restrict__ bx, Ray ray) {
    const float nan = __int_as_float(0x7fffffff);
    const float4 a0 = ldg4(bx), a1 = ldg4(bx + 1), a2 = ldg4(bx + 2), hi = ldg4(bx + 3);
    float t_in = -__int_as_float(0x7f800000), t_out = __int_as_float(0x7f800000);
    auto slab = [&](float4 a, float h) -> bool {
        const float dn = dot(v3(a), ray.d), on = dot(v3(a), ray.o);
        if (fabsf(dn) < 1e-8f) return on >= a.w && on <= h;
        const float inv = __fdividef(1.0f, dn);
        const float ta = (a.w - on) * inv, tb = (h - on) * inv;
        t_in = fmaxf(t_in, fminf(ta, tb));
        t_out = fminf(t_out, fmaxf(ta, tb));
        return true;
    };
    if (!slab(a0, hi.x) || !slab(a1, hi.y) || !slab(a2, hi.z)) return make_float2(nan, nan);
    if (!(t_in <= t_out) || !(t_out > t_in + 0.0001f)) return make_float2(nan, nan);
    return make_float2(t_in, t_out);
}

// constant_medium.h:20-53 for every medium, against the closest surface hit so far.
// Returns the index of the medium that scattered the ray (or -1) and updates t_hit.
// A boundary that is one static sphere (both media of the book-2 scene) takes ONE quadratic:
// sphere::hit over the universe returns the smaller root, and over (t1 + 1e-4, inf) the larger
// one if it lies beyond t1 + 1e-4 (sphere.h:44-49).
// GENERAL = false: every boundary of the scene is one static sphere (both media of C5); the out-of-line box / generic
// paths are then not even call sites -- they cost the caller registers and spills where they never run (C5 +3.7 %).
template <bool STATS, bool GENERAL>
__device__ __forceinline__ int media_hit(const DevScene& S, const Ray& ray, float tmin, float& t_hit, const Rng& rng,
                                         uint32_t bounce, Stats* st) {
    int which = -1;
    const float a = dot(ray.d, ray.d);
    // 1/|d| from one MUFU.RSQ and the free-flight logarithm from one MUFU.LG2 (errors ~1e-7 relative
    // and ~1e-7 absolute: far inside the Monte Carlo noise of a scattering distance) instead of an
    // IEEE division, a square root, a second division and logf: this runs for every ray of a scene
    // with media, +2.6 % on C5
    const float inv_len = rsqrtf(a);
    const float inv_a = inv_len * inv_len;
    const float ray_length = a * inv_len;
    float4 u4 = make_float4(0, 0, 0, 0);
    for (int m = 0; m < S.n_media; m++) {
        if ((m & 3) == 0) u4 = rng.draw(bounce, RS_MEDIUM + (m >> 2));
        float u = (m & 3) == 0 ? u4.x : ((m & 3) == 1 ? u4.y : ((m & 3) == 2 ? u4.z : u4.w));
        const DevMedium& md = S.media[m];
        if (STATS) { st->medium_queries++; st->boundary_tests += md.box >= 0 ? 1 : 2 * md.bcount; }  // a box boundary is one three-slab test
        float t1, t2;
        if (md.sphere >= 0) {
            float4 s = ldg4(S.sph + md.sphere);
            V3 oc = v3(s) - ray.o;
            float k = dot(ray.d, oc) * inv_a;
            float r2 = s.w * s.w;
            float cterm = dot(oc, oc) - r2;
            if (fabsf(cterm) < 0.125f * r2) {
                const float2 roots = sphere_roots_fp64(S.sph_d + 4 * (size_t)md.sphere, false, ray);  // NaN: fails the test below
                t1 = roots.x;
                t2 = roots.y;
            } else {
                V3 l = fma3(-k, ray.d, oc);
                float disc = r2 - dot(l, l);
                if (disc < 0.0f) continue;
                float sq = sqrtf(disc * inv_a);
                t1 = k - sq;
                t2 = k + sq;
            }
            if (!(t2 > t1 + 0.0001f)) continue;
        } else if (!GENERAL) {
            continue;  // instance for scenes whose boundaries are all single spheres: no call site of the two below
        } else {
            const float2 tt = md.box >= 0 ? boundary_pair_box(S.media_box + 4 * (size_t)md.box, ray)
                                          : boundary_pair_generic(S, md.bfirst, md.bcount, ray, inv_a);
            if (isnan(tt.x)) continue;
            t1 = tt.x;
            t2 = tt.y;
        }
        if (t1 < tmin) t1 = tmin;
        if (t2 > t_hit) t2 = t_hit;
        if (t1 >= t2) continue;
        if (t1 < 0.0f) t1 = 0.0f;
        float distance_inside = (t2 - t1) * ray_length;
        float hit_distance = md.neg_inv_density * __logf(u);
        if (hit_distance > distance_inside) continue;
        t_hit = fmaf(hit_distance, inv_len, t1);
        which = m;
    }
    return which;
}

// ---------------------------------------------------------------------------------
// textures (texture.h) and Perlin noise (perlin.h)
// ---------------------------------------------------------------------------------
// perlin.h:14-37.  FP32 throughout, and EXACT where it matters: the octave scaling p * 2^k only changes the exponent,
// floorf of a float is a float, and px - floorf(px) needs no more bits than px has, so the lattice cell and the
// fractional position are the same numbers a double-precision split of the same (FP32) point would give -- without the
// FP64 conversions the first version spent on it (3.3 % of C5's time at 2.4 lanes for ONE marble sphere).
__device__ __forceinline__ float perlin_noise(const DevScene& S, int pidx, float px, float py, float pz) {
    const float4* vec = S.perlin_vec + 256 * (size_t)pidx;
    const unsigned char* perm = S.perlin_perm + 768 * (size_t)pidx;
    const float fx = floorf(px), fy = floorf(py), fz = floorf(pz);
    const float u = px - fx, v = py - fy, w = pz - fz;
    // the lattice index modulo 256 (perlin.h:25-27 `& 255`): beyond 2^31 the float is a multiple of 256 anyway
    const int i = fabsf(fx) < 2.0e9f ? (int)fx : 0, j = fabsf(fy) < 2.0e9f ? (int)fy : 0, k = fabsf(fz) < 2.0e9f ? (int)fz : 0;
    float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
    float accum = 0.0f;
    // the corners one at a time, in the same order: unrolled, their eight gathers were in flight together, and the
    // registers that took raised what every caller of tex_value_general has to save around the call
#pragma unroll 1
    for (int di = 0; di < 2; di++)
#pragma unroll 1
        for (int dj = 0; dj < 2; dj++)
#pragma unroll 1
            for (int dk = 0; dk < 2; dk++) {
                int h = __ldg(perm + ((i + di) & 255)) ^ __ldg(perm + 256 + ((j + dj) & 255)) ^ __ldg(perm + 512 + ((k + dk) & 255));
                float4 g = __ldg(vec + h);
                float wx = u - di, wy = v - dj, wz = w - dk;
                accum += (di ? uu : 1.0f - uu) * (dj ? vv : 1.0f - vv) * (dk ? ww : 1.0f - ww) * (g.x * wx + g.y * wy + g.z * wz);
            }
    return accum;
}

__device__ __forceinline__ float perlin_turb(const DevScene& S, int pidx, V3 p, int depth) {
    float accum = 0.0f, weight = 1.0f;
    float x = p.x, y = p.y, z = p.z;
    for (int i = 0; i < depth; i++) {
        accum += weight * perlin_noise(S, pidx, x, y, z);
        weight *= 0.5f;
        x *= 2.0f; y *= 2.0f; z *= 2.0f;
    }
    return fabsf(accum);
}

__device__ __forceinline__ void sphere_uv(V3 n, float& u, float& v) {  // sphere.h:67-73
    const float pi = 3.14159265358979323846f;
    float theta = acosf(fminf(fmaxf(-n.y, -1.0f), 1.0f));
    float phi = atan2f(-n.z, n.x) + pi;
    u = phi / (2.0f * pi);
    v = theta / pi;
}

// uv_xf > -2: the hit is on a sphere whose (u, v) have not been computed: `outward` is its outward unit normal and
// uv_xf its transform (-1 none).  sphere.h:67-73 (an acos, an atan2 and a rotation back to object space) then runs HERE,
// out of line and only for the textures that read (u, v) -- the hot kernel body carries none of it (instruction cache).
__device__ __noinline__ V3 tex_value_general(const DevScene& S, int tex, float u, float v, V3 p, int uv_xf, V3 outward) {
    auto resolve_uv = [&]() {
        if (uv_xf <= -2) return;
        V3 n = outward;
        if (uv_xf >= 0) {  // back to object space: R^T n
            const float* R = S.xrot + 9 * (size_t)uv_xf;
            n = v3(R[0] * outward.x + R[3] * outward.y + R[6] * outward.z, R[1] * outward.x + R[4] * outward.y + R[7] * outward.z,
                   R[2] * outward.x + R[5] * outward.y + R[8] * outward.z);
        }
        sphere_uv(n, u, v);
        uv_xf = -2;
    };
    // checker textures select a child and recurse (texture.h:42-50, 66-76): iterate instead
    for (int level = 0; level < 16; level++) {
        const DevTexture& t = S.texs[tex];
        if (t.type == RT_TEX_SOLID) {
            return v3(t.color);
        } else if (t.type == RT_TEX_CHECKER) {
            int xi = (int)floorf(t.scale * p.x), yi = (int)floorf(t.scale * p.y), zi = (int)floorf(t.scale * p.z);
            tex = ((xi + yi + zi) % 2 == 0) ? t.a : t.b;
        } else if (t.type == RT_TEX_CHECKER_TRIANGLE) {
            resolve_uv();
            v = 1.0f - v;  // texture.h:68: flipped, and the flipped value is what the child sees
            int ui = (int)roundf(t.scale * u * 10.0f), vi = (int)roundf(t.scale * v * 10.0f);
            tex = ((ui + vi) % 2 == 0) ? t.a : t.b;
        } else if (t.type == RT_TEX_IMAGE) {
            if (t.a < 0) return v3(0.0f, 1.0f, 1.0f);  // texture.h:92
            resolve_uv();
            const DevImage& im = S.images[t.a];
            float uc = fminf(fmaxf(u, 0.0f), 1.0f);
            float vc = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
            int i = (int)(uc * im.w), j = (int)(vc * im.h);
            i = i < 0 ? 0 : (i < im.w ? i : im.w - 1);  // rtw_stb_image.h:83-88
            j = j < 0 ? 0 : (j < im.h ? j : im.h - 1);
            const unsigned char* px = im.rgb + 3 * ((size_t)j * im.w + i);
            const float s = 1.0f / 255.0f;
            return v3(s * __ldg(px), s * __ldg(px + 1), s * __ldg(px + 2));
        } else {  // noise: texture.h:115
            float turb = perlin_turb(S, t.a, p, 7);
            float val = 0.5f * (1.0f + sinf(fmaf(t.scale, p.z, 10.0f * turb)));
            return v3(val, val, val);
        }
    }
    return v3(0, 0, 0);
}

// solid_color is by far the most common texture: keep it inline, send the rest out of line
__device__ __forceinline__ V3 tex_value(const DevScene& S, int tex, float u, float v, V3 p, int uv_xf = -2, V3 outward = V3{0.0f, 0.0f, 0.0f}) {
    const DevTexture& t = S.texs[tex];
    if (t.type == RT_TEX_SOLID) return v3(t.color);
    return tex_value_general(S, tex, u, v, p, uv_xf, outward);
}

// ---------------------------------------------------------------------------------
// hit record completion + materials (material.h)
// ---------------------------------------------------------------------------------
struct Surface {
    float t;
    V3 p, normal;
    float u, v;
    int material;
    int prim_id;
    int nee_light;  // > 0: this surface is emitter number nee_light - 1 of the next-event list
    int uv_xf = -2;  // -2: (u, v) are valid; >= -1: a sphere hit whose (u, v) the texture lookup computes on demand (its transform)
    bool front;
};

// The accepted sphere hit re-solved in double (sphere.h:33-52 verbatim); out of line, once per
// sphere hit.  Ray in and result out by value, for the reason given at sphere_roots_fp64.
struct RefinedHit {
    float t;
    V3 p, outward;
};
__device__ __noinline__ RefinedHit refine_sphere_hit(const double* __restrict__ cd, bool moving, Ray ray, float t_approx) {
    // the FP64 record is read HERE, not by the caller: the common FP32 completion then holds no doubles at all
    double cx = cd[0], cy = cd[1], cz = cd[2];
    const double rr = cd[3];
    if (moving) { cx += (double)ray.time * cd[4]; cy += (double)ray.time * cd[5]; cz += (double)ray.time * cd[6]; }
    double ox = cx - (double)ray.o.x, oy = cy - (double)ray.o.y, oz = cz - (double)ray.o.z;
    double dx = ray.d.x, dy = ray.d.y, dz = ray.d.z;
    double a = dx * dx + dy * dy + dz * dz;
    double hh = dx * ox + dy * oy + dz * oz;
    double cc = ox * ox + oy * oy + oz * oz - rr * rr;
    double sq = sqrt(fmax(hh * hh - a * cc, 0.0));
    double inv_a = 1.0 / a;
    double ta = (hh - sq) * inv_a, tb = (hh + sq) * inv_a;
    double td = fabs(ta - (double)t_approx) <= fabs(tb - (double)t_approx) ? ta : tb;
    double px = (double)ray.o.x + td * dx, py = (double)ray.o.y + td * dy, pz = (double)ray.o.z + td * dz;
    double inv_r = 1.0 / rr;
    RefinedHit r;
    r.t = (float)td;
    r.p = v3((float)px, (float)py, (float)pz);
    r.outward = v3((float)((px - cx) * inv_r), (float)((py - cy) * inv_r), (float)((pz - cz) * inv_r));  // sphere.h:52
    return r;
}

// LITE / MSPH as in hit_prim: the instance for scenes without triangles / without moving spheres has none of their code.
template <bool LITE = false, bool MSPH = true>
__device__ __forceinline__ void complete_hit(const DevScene& S, const Ray& ray, const Hit& hit, Surface& sf, bool want_uv) {
    uint32_t type = hit.prim >> 28, idx = hit.prim & 0x0fffffffu;
    sf.t = hit.t;
    sf.p = fma3(hit.t, ray.d, ray.o);
    V3 outward;
    sf.u = hit.u;
    sf.v = hit.v;
    sf.nee_light = 0;
    if (type == PT_SPHERE || type == PT_MSPHERE) {
        // The accepted sphere hit is re-solved ONCE in double (sphere.h:33-52 verbatim): the
        // FP32 traversal fixes WHICH root of WHICH sphere, the FP64 pass fixes t, p and the
        // normal, so that a far-away small sphere still gets a normal good to FP32 rounding.
        int4 sh;
        float4 s;          // centre and radius in FP32 (the device record the traversal tested)
        const double* cd;  // the same in double, read only by the refinement
        const bool moving = MSPH && type != PT_SPHERE;
        if (!moving) {
            s = ldg4(S.sph + idx);
            cd = S.sph_d + 4 * (size_t)idx;
            sh = __ldg(S.sph_sh + idx);
        } else {
            const float4* m = S.msph + 2 * (size_t)idx;
            const float4 a = ldg4(m), b = ldg4(m + 1);
            const V3 c = fma3(ray.time, v3(b), v3(a));  // sphere.h:33 center.at(r.time())
            s = make_float4(c.x, c.y, c.z, a.w);
            cd = S.msph_d + 8 * (size_t)idx;
            sh = __ldg(S.msph_sh + idx);
        }
        // FP32 suffices unless the sphere is small relative to its distance (the FP32 hit point is
        // only good to ulp(|p|), which the normal magnifies by 1/r) or the ray starts near the
        // surface of a big sphere (cancellation in |oc|^2 - r^2)
        {
            V3 oc = v3(s) - ray.o;
            float oc2 = dot(oc, oc), r2 = s.w * s.w;
            if (want_uv || oc2 > 64.0f * r2 || fabsf(oc2 - r2) < 0.125f * r2) {
                const RefinedHit r = refine_sphere_hit(cd, moving, ray, hit.t);
                sf.t = r.t;
                sf.p = r.p;
                outward = r.outward;
            } else {
                outward = __frcp_rn(s.w) * (sf.p - v3(s));  // sphere.h:52
            }
        }
        sf.material = sh.x;
        sf.prim_id = sh.z;
        sf.u = sf.v = 0.0f;
        sf.uv_xf = sh.y < 0 ? -1 : sh.y;  // (u, v) on demand: tex_value_general
        if (want_uv) {                    // the probes want them here
            V3 n = outward;
            if (sh.y >= 0) {  // back to object space: R^T n
                const float* R = S.xrot + 9 * (size_t)sh.y;
                n = v3(R[0] * outward.x + R[3] * outward.y + R[6] * outward.z,
                       R[1] * outward.x + R[4] * outward.y + R[7] * outward.z,
                       R[2] * outward.x + R[5] * outward.y + R[8] * outward.z);
            }
            sphere_uv(n, sf.u, sf.v);
            sf.uv_xf = -2;
        }
    } else if (LITE || type == PT_QUAD) {
        outward = v3(ldg4(S.quad + 3 * (size_t)idx));
        int4 sh = __ldg(S.quad_sh + idx);
        sf.material = sh.x;
        sf.prim_id = sh.z;
        sf.nee_light = sh.w;
    } else {
        const float4* ts = S.tri_sh + 3 * (size_t)idx;
        float4 a = ldg4(ts), b = ldg4(ts + 1), c = ldg4(ts + 2);
        outward = v3(a);
        sf.material = __float_as_int(a.w);
        sf.prim_id = __float_as_int(c.z);
        float alpha = 1.0f - hit.u - hit.v, beta = hit.u, gamma = hit.v;  // triangle.h:96-104
        sf.u = alpha * b.x + beta * b.z + gamma * c.x;
        sf.v = alpha * b.y + beta * b.w + gamma * c.y;
    }
    sf.front = dot(ray.d, outward) < 0.0f;  // hittable.h:22-25
    sf.normal = sf.front ? outward : -outward;
}

// The accepted hit of a DETERMINISTIC ray (primary-hit AOV, probe rays) completed in double from the
// double-precision ray: the FP32 traversal decides WHICH primitive (and which sphere root), this pass
// restates the reference's own arithmetic for t, p, normal and uv (sphere.h:33-58, quad.h:30-47 with the
// planar coordinates as dot products, triangle.h:67-110) on the FP64 copies of the records, so that the
// parity gate compares values good to FP32 rounding of the RESULT (north_star: t and normal within 1e-5).
// Out of line; the render kernels never call it (their rays are FP32 by construction).
struct RayD {
    double o[3], d[3], time;
};
__device__ __noinline__ void complete_hit_fp64(const DevScene& S, const RayD& r, const Hit& hit, Surface& sf) {
    const uint32_t type = hit.prim >> 28, idx = hit.prim & 0x0fffffffu;
    const double ox = r.o[0], oy = r.o[1], oz = r.o[2], dx = r.d[0], dy = r.d[1], dz = r.d[2];
    double t, nx, ny, nz;
    sf.nee_light = 0;
    sf.u = sf.v = 0.0f;
    if (type == PT_SPHERE || type == PT_MSPHERE) {
        double cx, cy, cz, rr;
        int4 sh;
        if (type == PT_SPHERE) {
            const double* cd = S.sph_d + 4 * (size_t)idx;
            cx = cd[0]; cy = cd[1]; cz = cd[2]; rr = cd[3];
            sh = __ldg(S.sph_sh + idx);
        } else {
            const double* cd = S.msph_d + 8 * (size_t)idx;
            cx = cd[0] + r.time * cd[4]; cy = cd[1] + r.time * cd[5]; cz = cd[2] + r.time * cd[6];
            rr = cd[3];
            sh = __ldg(S.msph_sh + idx);
        }
        const double qx = cx - ox, qy = cy - oy, qz = cz - oz;
        const double a = dx * dx + dy * dy + dz * dz;
        const double hh = dx * qx + dy * qy + dz * qz;
        const double cc = qx * qx + qy * qy + qz * qz - rr * rr;
        const double sq = sqrt(fmax(hh * hh - a * cc, 0.0));
        const double ta = (hh - sq) / a, tb = (hh + sq) / a;
        t = fabs(ta - (double)hit.t) <= fabs(tb - (double)hit.t) ? ta : tb;
        const double px = ox + t * dx, py = oy + t * dy, pz = oz + t * dz;
        nx = (px - cx) / rr; ny = (py - cy) / rr; nz = (pz - cz) / rr;  // sphere.h:52
        sf.material = sh.x;
        sf.prim_id = sh.z;
        double ux = nx, uy = ny, uz = nz;
        if (sh.y >= 0) {  // back to object space: R^T n
            const float* R = S.xrot + 9 * (size_t)sh.y;
            ux = R[0] * nx + R[3] * ny + R[6] * nz;
            uy = R[1] * nx + R[4] * ny + R[7] * nz;
            uz = R[2] * nx + R[5] * ny + R[8] * nz;
        }
        const double pi = 3.1415926535897932385;  // sphere.h:67-73
        sf.u = (float)((atan2(-uz, ux) + pi) / (2.0 * pi));
        sf.v = (float)(acos(fmin(fmax(-uy, -1.0), 1.0)) / pi);
    } else if (type == PT_QUAD) {
        const double* q = S.quad_d + 12 * (size_t)idx;
        nx = q[0]; ny = q[1]; nz = q[2];
        t = (q[3] - (nx * ox + ny * oy + nz * oz)) / (nx * dx + ny * dy + nz * dz);
        const double px = ox + t * dx, py = oy + t * dy, pz = oz + t * dz;
        sf.u = (float)(q[4] * px + q[5] * py + q[6] * pz - q[7]);
        sf.v = (float)(q[8] * px + q[9] * py + q[10] * pz - q[11]);
        const int4 sh = __ldg(S.quad_sh + idx);
        sf.material = sh.x;
        sf.prim_id = sh.z;
        sf.nee_light = sh.w;
    } else {
        const double* td = S.tri_d + 9 * (size_t)idx;
        const double e1x = td[3], e1y = td[4], e1z = td[5], e2x = td[6], e2y = td[7], e2z = td[8];
        const double pvx = dy * e2z - dz * e2y, pvy = dz * e2x - dx * e2z, pvz = dx * e2y - dy * e2x;
        const double inv = 1.0 / (e1x * pvx + e1y * pvy + e1z * pvz);
        const double tx = ox - td[0], ty = oy - td[1], tz = oz - td[2];
        const double bu = (tx * pvx + ty * pvy + tz * pvz) * inv;
        const double qx = ty * e1z - tz * e1y, qy = tz * e1x - tx * e1z, qz = tx * e1y - ty * e1x;
        const double bv = (dx * qx + dy * qy + dz * qz) * inv;
        t = (e2x * qx + e2y * qy + e2z * qz) * inv;
        const float4* ts = S.tri_sh + 3 * (size_t)idx;
        const float4 a = ldg4(ts), b = ldg4(ts + 1), c = ldg4(ts + 2);
        // the unit normal from the FP64 edges (triangle.h:21-22)
        const double cxn = e1y * e2z - e1z * e2y, cyn = e1z * e2x - e1x * e2z, czn = e1x * e2y - e1y * e2x;
        const double il = 1.0 / sqrt(cxn * cxn + cyn * cyn + czn * czn);
        nx = cxn * il; ny = cyn * il; nz = czn * il;
        sf.material = __float_as_int(a.w);
        sf.prim_id = __float_as_int(c.z);
        const double alpha = 1.0 - bu - bv;  // triangle.h:96-104
        sf.u = (float)(alpha * b.x + bu * b.z + bv * c.x);
        sf.v = (float)(alpha * b.y + bu * b.w + bv * c.y);
    }
    sf.t = (float)t;
    sf.p = v3((float)(ox + t * dx), (float)(oy + t * dy), (float)(oz + t * dz));
    sf.front = dx * nx + dy * ny + dz * nz < 0.0;  // hittable.h:22-25
    sf.normal = sf.front ? v3((float)nx, (float)ny, (float)nz) : v3((float)-nx, (float)-ny, (float)-nz);
}

// vec3.h:107-115: the `1e-160 < lensq <= 1` test is always true, so this is
// normalise(uniform point of the cube [-1,1]^3) with no rejection (SURVEY Q1).
__device__ __forceinline__ V3 random_unit_vector(float ux, float uy, float uz) {
    V3 p = v3(fmaf(2.0f, ux, -1.0f), fmaf(2.0f, uy, -1.0f), fmaf(2.0f, uz, -1.0f));
    float lensq = dot(p, p);
    return rsqrtf(lensq) * p;
}
__device__ __forceinline__ V3 reflect(V3 v, V3 n) { return v - 2.0f * dot(v, n) * n; }
__device__ __forceinline__ bool near_zero(V3 v) { return fabsf(v.x) < 1e-8f && fabsf(v.y) < 1e-8f && fabsf(v.z) < 1e-8f; }

// The author's `specular` material (material.h:145-167).  Out of line: powf alone is ~150
// instructions and the material appears in one scene.
__device__ __noinline__ V3 specular_direction(V3 unit, V3 refl, V3 ruv, V3 normal, float shininess) {
    V3 diffuse = ruv;  // random_on_hemisphere (vec3.h:116-124)
    if (!(dot(diffuse, normal) > 0.0f)) diffuse = -diffuse;
    float factor = powf(1.0f - dot(refl, unit), shininess);
    V3 dir = factor * refl + (1.0f - factor) * diffuse;
    if (near_zero(dir)) dir = normal;
    return dir;
}

// material::emitted (material.h:14,99-101,111-113) and material::scatter (material.h:29-38,
// 47-74, 82-88, 129-134, 145-167) of one hit.  `draw_u4()` returns the uniforms of this bounce (see Rng); it is called
// after the texture lookup, only for a material that scatters, so the four uniforms are not live across the call of
// tex_value_general.
// Returns false when the path ends here (absorbed, or a light).  Written so that the five
// materials share what they have in common -- the texture lookup, the unit vector of
// vec3.h:107-115, the normalised incoming direction and its mirror image -- and differ in a
// handful of instructions each: the material switch is the most divergent code of the shade
// phase, and its size is instruction-cache footprint.
// SPECULAR = false: no material of the scene is RT_MAT_SPECULAR (the reference's `specular` class, unused by its own
// scenes): no call site of specular_direction.
template <bool SPECULAR = true, class DrawU4>
__device__ __forceinline__ bool shade_surface(const DevScene& S, const DevMaterial& m, const Ray& in, const Surface& sf, DrawU4 draw_u4,
                                              V3& emitted, V3& attenuation, Ray& out) {
    out.o = sf.p;
    out.time = in.time;
    out.d = sf.normal;
    V3 texc = v3(0, 0, 0);
    if (m.tex >= 0) texc = tex_value(S, m.tex, sf.u, sf.v, sf.p, sf.uv_xf, sf.front ? sf.normal : -sf.normal);
    emitted = v3(0, 0, 0);
    attenuation = texc;
    if (m.type == RT_MAT_DIFFUSE_LIGHT || m.type == RT_MAT_EMISSIVE_LIGHT) {  // material.h:17-19, 99-101, 116-118
        emitted = texc;
        return false;
    }
    const float4 u4 = draw_u4();
    const V3 ruv = random_unit_vector(u4.x, u4.y, u4.z);
    if (m.type == RT_MAT_LAMBERTIAN) {  // the common case first, with nothing it does not need
        V3 dir = sf.normal + ruv;
        if (near_zero(dir)) dir = sf.normal;
        out.d = dir;
        return true;
    }
    if (m.type == RT_MAT_ISOTROPIC) {
        out.d = ruv;
        return true;
    }
    const V3 unit = normalize(in.d);
    const float cos_in = dot(unit, sf.normal);
    const V3 refl = unit - (2.0f * cos_in) * sf.normal;  // reflect(unit, n), vec3.h:125-127
    attenuation = v3(m.albedo);
    if (m.type == RT_MAT_METAL) {
        // unit_vector(reflect(d, n)) == reflect(unit_vector(d), n) (material.h:83-84)
        V3 dir = fma3(m.param, ruv, normalize(refl));
        out.d = dir;
        return dot(dir, sf.normal) > 0.0f;
    }
    if (m.type == RT_MAT_DIELECTRIC) {
        attenuation = v3(1.0f, 1.0f, 1.0f);
        const float ri = sf.front ? __fdividef(1.0f, m.param) : m.param;
        const float cos_theta = fminf(-cos_in, 1.0f);
        const float sin_theta = sqrtf(fmaxf(1.0f - cos_theta * cos_theta, 0.0f));
        float r0 = __fdividef(1.0f - ri, 1.0f + ri);
        r0 = r0 * r0;
        const float x = 1.0f - cos_theta;
        const float reflectance = r0 + (1.0f - r0) * (x * x) * (x * x) * x;
        if (ri * sin_theta > 1.0f || reflectance > u4.w) {
            out.d = refl;
        } else {  // vec3.h:128-133
            V3 perp = ri * (unit + cos_theta * sf.normal);
            V3 para = -sqrtf(fabsf(1.0f - dot(perp, perp))) * sf.normal;
            out.d = perp + para;
        }
        return true;
    }
    if (SPECULAR) out.d = specular_direction(unit, refl, ruv, sf.normal, m.param);  // RT_MAT_SPECULAR
    return true;
}

// kept for the probes and the first kernel version: the same thing in two calls
__device__ __forceinline__ V3 mat_emitted(const DevScene& S, const DevMaterial& m, const Surface& sf) {
    if (m.type == RT_MAT_DIFFUSE_LIGHT || m.type == RT_MAT_EMISSIVE_LIGHT) return tex_value(S, m.tex, sf.u, sf.v, sf.p, sf.uv_xf, sf.front ? sf.normal : -sf.normal);
    return v3(0, 0, 0);
}
__device__ __forceinline__ bool mat_scatter(const DevScene& S, const DevMaterial& m, const Ray& in, const Surface& sf, float4 u4,
                                            V3& attenuation, Ray& out) {
    V3 emitted;
    return shade_surface(S, m, in, sf, [&] { return u4; }, emitted, attenuation, out);
}

// Camera.txt:240-272: unshadowed point lights
__device__ __noinline__ V3 point_lighting(const DevScene& S, V3 p, V3 normal) {
    V3 result = v3(0, 0, 0);
    for (int i = 0; i < S.n_lights; i++) {
        const DevLight& l = S.lights[i];
        V3 ld = v3(l.pos) - p;
        float d2 = dot(ld, ld);
        ld = (1.0f / sqrtf(d2)) * ld;
        float diffuse = fmaxf(dot(normal, ld), 0.0f);
        if (d2 <= l.size * l.size) {
            result = result + diffuse * v3(l.intensity);
        } else {
            float att = 1.0f / (d2 + l.size * 0.1f);
            result = result + (diffuse * att) * v3(l.intensity);
        }
    }
    return result;
}

// ---------------------------------------------------------------------------------
// Next-event estimation (opt-in, RT_FLAG_NEE; SURVEY 8f rank 4).
//
// The reference estimates L_o = albedo * L_i(w) with ONE direction w drawn from its own
// sampler: w = n + unit(c), c uniform in the cube [-1,1]^3 (vec3.h:107-115, SURVEY Q1) for a
// lambertian, w = unit(c) for the isotropic phase function.  The expectation is split here into
// the part that comes straight from the quad emitters -- estimated by sampling a point ON an
// emitter and weighting with the density p(w) of the reference's sampler -- and the rest, for which
// the scattered ray goes on as before but does not collect the emission of a listed emitter it hits
// next.  Same expectation (the converged image is the reference's), much less variance where the
// emitters are small.  The two ways of finding an emitter -- the sampled point and the scattered ray
// that happens to hit it -- are combined with the balance heuristic (weights p_light / (p_light +
// p_w) and p_w / (p_light + p_w), both densities per steradian), which keeps the light sample's
// 1 / r^2 bounded for vertices close to an emitter (the Cornell ceiling is one unit above its light).  Density of unit(c) on the sphere: (1/8) * integral_0^R r^2 dr = R^3 / 24 per
// steradian, R = 1 / max|u_i| the distance to the cube's face; w = unit(n + u) maps the unit
// sphere around n to directions with dA_u = 4 cos(theta) dw, so p_lambert(w) = R(u)^3 cos(theta) / 6
// with u = 2 cos(theta) w - n (for a uniform u this is the cosine lobe cos/pi).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ float cube_point_density(V3 u) {  // of unit(c), per steradian
    const float m = fmaxf(fabsf(u.x), fmaxf(fabsf(u.y), fabsf(u.z)));
    const float R = 1.0f / m;
    return R * R * R * (1.0f / 24.0f);
}
// density of the reference's scattering direction `dir` (unit) at a vertex with normal n
__device__ __forceinline__ float scatter_density(V3 dir, V3 n, bool isotropic) {
    if (isotropic) return cube_point_density(dir);
    const float c = dot(dir, n);
    if (!(c > 0.0f)) return 0.0f;
    return cube_point_density((2.0f * c) * dir - n) * 4.0f * c;
}
// density per steradian with which the emitter sampler proposes the point at squared distance r2 seen under cos_y
__device__ __forceinline__ float light_density(const DevScene& S, float r2, float cos_y) { return r2 / (cos_y * S.nee_total_area); }

// Probability that a ray survives every constant_medium between tmin and tmax (constant_medium.h:20-53:
// the free-flight distance is exponential with rate density, times the leaf multiplicity of Q15).
__device__ __forceinline__ float media_transmittance(const DevScene& S, const Ray& ray, float tmin, float tmax) {
    const float a = dot(ray.d, ray.d);
    const float inv_a = 1.0f / a;
    const float ray_length = sqrtf(a);
    float optical_depth = 0.0f;
    for (int m = 0; m < S.n_media; m++) {
        const DevMedium& md = S.media[m];
        float t1, t2;
        if (md.sphere >= 0) {
            float4 s = ldg4(S.sph + md.sphere);
            V3 oc = v3(s) - ray.o;
            float k = dot(ray.d, oc) * inv_a;
            float r2 = s.w * s.w;
            float cterm = dot(oc, oc) - r2;
            if (fabsf(cterm) < 0.125f * r2) {
                const float2 roots = sphere_roots_fp64(S.sph_d + 4 * (size_t)md.sphere, false, ray);  // NaN: fails the test below
                t1 = roots.x;
                t2 = roots.y;
            } else {
                V3 l = fma3(-k, ray.d, oc);
                float disc = r2 - dot(l, l);
                if (disc < 0.0f) continue;
                float sq = sqrtf(disc * inv_a);
                t1 = k - sq;
                t2 = k + sq;
            }
            if (!(t2 > t1 + 0.0001f)) continue;
        } else {
            const float2 tt = md.box >= 0 ? boundary_pair_box(S.media_box + 4 * (size_t)md.box, ray)
                                          : boundary_pair_generic(S, md.bfirst, md.bcount, ray, inv_a);
            if (isnan(tt.x)) continue;
            t1 = tt.x;
            t2 = tt.y;
        }
        if (t1 < tmin) t1 = tmin;
        if (t2 > tmax) t2 = tmax;
        if (t1 >= t2) continue;
        if (t1 < 0.0f) t1 = 0.0f;
        optical_depth += (t2 - t1) * ray_length * (-1.0f / md.neg_inv_density);
    }
    return __expf(-optical_depth);
}

// shadow rays go through whichever acceleration structure the kernel instance traverses
// (traverse_wide is defined in rt_wide.cuh)
template <int W, bool STATS>
__device__ __forceinline__ void traverse_wide(const DevScene& S, const Ray& ray, float tmin, float tmax, uint32_t origin_prim, Hit& hit,
                                              Stats* st);
template <int WIDTH>
__device__ __forceinline__ void traverse_sel(const DevScene& S, const Ray& ray, float tmin, float tmax, uint32_t origin_prim, Hit& hit) {
    if constexpr (WIDTH == 2) {
        traverse(S, ray, tmin, tmax, origin_prim, hit);
    } else {
        traverse_wide<WIDTH, false>(S, ray, tmin, tmax, origin_prim, hit, nullptr);
    }
}

// The directly-lit part of one lambertian / isotropic scattering event at p: radiance per unit of
// (throughput * albedo).  `u` = three uniforms (which emitter, where on it).
template <int WIDTH>
__device__ __noinline__ V3 nee_direct(const DevScene& S, V3 p, V3 n, bool isotropic, uint32_t origin_prim, float time, float4 u) {
    int k = 0;
    while (k + 1 < S.n_nee_lights && u.x >= S.nee_lights[k].cdf) k++;
    const DevNeeLight& lt = S.nee_lights[k];
    const V3 y = v3(lt.Q) + u.y * v3(lt.u) + u.z * v3(lt.v);
    const V3 w = y - p;
    const float r2 = dot(w, w);
    if (!(r2 > 0.0f)) return v3(0, 0, 0);
    const float r = sqrtf(r2);
    const V3 dir = (1.0f / r) * w;
    const float density = scatter_density(dir, n, isotropic);
    if (!(density > 0.0f)) return v3(0, 0, 0);
    const float cos_y = fabsf(dot(dir, v3(lt.n)));  // diffuse_light emits from both faces (material.h:99-101)
    if (!(cos_y > 0.0f)) return v3(0, 0, 0);
    Ray sray;
    sray.o = p;
    sray.d = dir;
    sray.time = time;
    const float tmax = r * (1.0f - 1e-4f);
    Hit h;
    traverse_sel<WIDTH>(S, sray, 0.001f, tmax, origin_prim, h);
    if (h.prim != PRIM_NONE) return v3(0, 0, 0);
    // Le * p_w / p_light, times the balance-heuristic weight p_light / (p_light + p_w)
    float weight = density / (light_density(S, r2, cos_y) + density);
    if (S.n_media > 0) weight *= media_transmittance(S, sray, 0.001f, tmax);
    return weight * tex_value(S, lt.tex, u.y, u.z, y);
}

// Camera.txt:240-272 with the one thing the reference leaves out: a shadow ray per light
// (RT_FLAG_SHADOWED_POINT_LIGHTS, opt-in -- it changes the image on purpose: the reference's
// point lights shine through everything).  Media on the way attenuate the light as well.
template <int WIDTH>
__device__ __noinline__ V3 point_lighting_shadowed(const DevScene& S, V3 p, V3 normal, uint32_t origin_prim, float time) {
    V3 result = v3(0, 0, 0);
    for (int i = 0; i < S.n_lights; i++) {
        const DevLight& l = S.lights[i];
        V3 ld = v3(l.pos) - p;
        const float d2 = dot(ld, ld);
        ld = (1.0f / sqrtf(d2)) * ld;
        const float diffuse = fmaxf(dot(normal, ld), 0.0f);
        if (!(diffuse > 0.0f)) continue;
        const float dist = sqrtf(d2);
        Ray sray;
        sray.o = p;
        sray.d = ld;
        sray.time = time;
        Hit h;
        traverse_sel<WIDTH>(S, sray, 0.001f, dist, origin_prim, h);
        if (h.prim != PRIM_NONE) continue;
        const float tm = S.n_media > 0 ? media_transmittance(S, sray, 0.001f, dist) : 1.0f;
        // the same arithmetic as point_lighting, so that an unoccluded light gives the same bits
        if (d2 <= l.size * l.size) {
            result = result + (tm * diffuse) * v3(l.intensity);
        } else {
            float att = 1.0f / (d2 + l.size * 0.1f);
            result = result + (tm * (diffuse * att)) * v3(l.intensity);
        }
    }
    return result;
}

// Camera.txt:177-200 get_ray.  Directions are built relative to the camera centre
// (dir00 = pixel00_loc - center, evaluated in double on the host) so that FP32 keeps
// sub-pixel accuracy when the camera sits hundreds of units from the origin.  `Cam` is anything with the camera fields
// of DevScene (center, dir00, du, dv, disk_u, disk_v, defocus): the scene itself, or one view of a multi-view batch,
// so both go through the same arithmetic.
template <bool LITE, class Cam>
__device__ __forceinline__ Ray camera_ray(const Cam& S, int i, int j, const Rng& rng) {
    float4 u = rng.draw(0, RS_CAMERA);
    float fx = (float)i + (u.x - 0.5f), fy = (float)j + (u.y - 0.5f);
    V3 dir = fma3(fx, v3(S.du), fma3(fy, v3(S.dv), v3(S.dir00)));
    Ray r;
    r.o = v3(S.center);
    r.time = u.z;
    if (!LITE && S.defocus) {
        // random_in_unit_disk (vec3.h:135-142): rejection sampling, two candidates per draw
        float px = 0.0f, py = 0.0f;
        for (uint32_t attempt = 0;; attempt++) {
            float4 c = rng.draw(0, RS_DEFOCUS + (attempt < 14 ? attempt : 14));
            px = fmaf(2.0f, c.x, -1.0f); py = fmaf(2.0f, c.y, -1.0f);
            if (px * px + py * py < 1.0f) break;
            px = fmaf(2.0f, c.z, -1.0f); py = fmaf(2.0f, c.w, -1.0f);
            if (px * px + py * py < 1.0f) break;
            if (attempt >= 14) { px = py = 0.0f; break; }  // (1 - pi/4)^30 ~ 1e-20
        }
        V3 off = fma3(px, v3(S.disk_u), py * v3(S.disk_v));
        r.o = r.o + off;
        dir = dir - off;
    }
    r.d = dir;
    return r;
}

}  // namespace rtdev
