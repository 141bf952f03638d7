// prim_derive.h — from one primitive of the C ABI (include/rt_b200.h) to its device records.
//
// Shared by the two scene-upload paths of rt_upload_scene: the host path (binned-SAH build,
// records written on the CPU) and the device path (csrc/bvh_device.cuh: LBVH build and record
// emission in CUDA kernels).  Everything here is arithmetic in double with ONE rounding per
// operation on both sides -- the device versions use __dmul_rn/__dadd_rn/__dsub_rn so that nvcc
// does not contract a*b+c into an FMA, and the host compiler targets baseline x86-64 (no FMA) --
// so both paths produce bit-identical records and therefore bit-identical images.
//
// Reference: sphere.h:12-30 (static / moving constructor), quad.h:13-21 (n, normal, D, w),
// triangle.h:16-30 (normal), hittable.h:39-146 (translate / rotate_y, baked here).
#pragma once
#include <cmath>
#include <cstdint>

#include "rt_b200.h"

#if defined(__CUDACC__)
#define RT_HD __host__ __device__
#else
#define RT_HD
#endif

namespace rtprep {

// device primitive types (the BVH leaf encoding stores them in 3 bits)
enum : uint32_t { PREP_SPHERE = 0, PREP_MSPHERE = 1, PREP_QUAD = 2, PREP_TRI = 3 };  // == PT_* of rt_device.cuh

RT_HD inline double dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
RT_HD inline double dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
RT_HD inline double dsub(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

struct D3 {
    double x, y, z;
};
RT_HD inline D3 d3(const double* p) { return D3{p[0], p[1], p[2]}; }
RT_HD inline D3 operator+(D3 a, D3 b) { return D3{dadd(a.x, b.x), dadd(a.y, b.y), dadd(a.z, b.z)}; }
RT_HD inline D3 operator-(D3 a, D3 b) { return D3{dsub(a.x, b.x), dsub(a.y, b.y), dsub(a.z, b.z)}; }
RT_HD inline D3 operator*(double s, D3 a) { return D3{dmul(s, a.x), dmul(s, a.y), dmul(s, a.z)}; }
RT_HD inline double ddot(D3 a, D3 b) { return dadd(dadd(dmul(a.x, b.x), dmul(a.y, b.y)), dmul(a.z, b.z)); }
RT_HD inline D3 dcross(D3 a, D3 b) {
    return D3{dsub(dmul(a.y, b.z), dmul(a.z, b.y)), dsub(dmul(a.z, b.x), dmul(a.x, b.z)), dsub(dmul(a.x, b.y), dmul(a.y, b.x))};
}
RT_HD inline D3 dunit(D3 a) { return (1.0 / sqrt(ddot(a, a))) * a; }

RT_HD inline D3 xf_point(const rt_xform* x, D3 p) {
    if (!x) return p;
    return D3{dadd(dadd(dadd(dmul(x->r[0], p.x), dmul(x->r[1], p.y)), dmul(x->r[2], p.z)), x->t[0]),
              dadd(dadd(dadd(dmul(x->r[3], p.x), dmul(x->r[4], p.y)), dmul(x->r[5], p.z)), x->t[1]),
              dadd(dadd(dadd(dmul(x->r[6], p.x), dmul(x->r[7], p.y)), dmul(x->r[8], p.z)), x->t[2])};
}
RT_HD inline D3 xf_dir(const rt_xform* x, D3 d) {
    if (!x) return d;
    return D3{dadd(dadd(dmul(x->r[0], d.x), dmul(x->r[1], d.y)), dmul(x->r[2], d.z)),
              dadd(dadd(dmul(x->r[3], d.x), dmul(x->r[4], d.y)), dmul(x->r[5], d.z)),
              dadd(dadd(dmul(x->r[6], d.x), dmul(x->r[7], d.y)), dmul(x->r[8], d.z))};
}

// One primitive with its instance transform applied (exact for rigid transforms).
struct BakedPrim {
    uint32_t dev_type;
    int prim_id;  // canonical id (-1 for boundaries)
    D3 a, b, c;   // sphere: c0, cvec, -; quad: Q, u, v; triangle: p0, p1, p2
    double radius;
    int material, xform;
    float uv[6];
};

// The typed source arrays of a scene description (host pointers on the host path, device copies
// on the device path; on the device path the mesh table points at device copies of the mesh arrays).
struct Sources {
    const rt_sphere* spheres;
    const rt_quad* quads;
    const rt_triangle* triangles;
    const rt_xform* xforms;
    const rt_mesh* meshes;
};

RT_HD inline BakedPrim bake_prim(const Sources& src, rt_prim_ref r, int prim_id) {
    BakedPrim b;
    b.prim_id = prim_id;
    b.radius = 0.0;
    b.c = D3{0, 0, 0};
    for (int k = 0; k < 6; k++) b.uv[k] = 0.0f;
    if (r.type == RT_PRIM_SPHERE) {
        const rt_sphere& s = src.spheres[r.index];
        const rt_xform* x = s.xform >= 0 ? &src.xforms[s.xform] : nullptr;
        b.a = xf_point(x, d3(s.center0));
        b.b = xf_dir(x, d3(s.center_vec));
        b.radius = s.radius;
        b.material = s.material;
        b.xform = s.xform;
        const bool moving = s.center_vec[0] != 0 || s.center_vec[1] != 0 || s.center_vec[2] != 0;
        b.dev_type = moving ? PREP_MSPHERE : PREP_SPHERE;
    } else if (r.type == RT_PRIM_QUAD) {
        const rt_quad& q = src.quads[r.index];
        const rt_xform* x = q.xform >= 0 ? &src.xforms[q.xform] : nullptr;
        b.a = xf_point(x, d3(q.Q));
        b.b = xf_dir(x, d3(q.u));
        b.c = xf_dir(x, d3(q.v));
        b.material = q.material;
        b.xform = q.xform;
        b.dev_type = PREP_QUAD;
    } else {
        const rt_triangle& t = src.triangles[r.index];
        const rt_xform* x = t.xform >= 0 ? &src.xforms[t.xform] : nullptr;
        b.a = xf_point(x, d3(t.p0));
        b.b = xf_point(x, d3(t.p1));
        b.c = xf_point(x, d3(t.p2));
        b.material = t.material;
        b.xform = t.xform;
        b.uv[0] = t.uv0[0]; b.uv[1] = t.uv0[1]; b.uv[2] = t.uv1[0]; b.uv[3] = t.uv1[1]; b.uv[4] = t.uv2[0]; b.uv[5] = t.uv2[1];
        b.dev_type = PREP_TRI;
    }
    return b;
}

// Triangle k of mesh `mesh` (indices already checked): the float positions widened to double, then
// transformed -- the same BakedPrim as an rt_triangle that holds the widened values.
RT_HD inline BakedPrim bake_mesh_triangle(const Sources& src, int mesh, uint32_t k, int prim_id) {
    const rt_mesh& m = src.meshes[mesh];
    const rt_xform* x = m.xform >= 0 ? &src.xforms[m.xform] : nullptr;
    const uint32_t* vi = m.indices + 3 * (size_t)k;
    const uint32_t* ti = m.uv_indices ? m.uv_indices + 3 * (size_t)k : vi;
    auto corner = [&](uint32_t v) {
        const float* p = m.positions + 3 * (size_t)v;
        return D3{(double)p[0], (double)p[1], (double)p[2]};
    };
    BakedPrim b;
    b.dev_type = PREP_TRI;
    b.prim_id = prim_id;
    b.radius = 0.0;
    b.a = xf_point(x, corner(vi[0]));
    b.b = xf_point(x, corner(vi[1]));
    b.c = xf_point(x, corner(vi[2]));
    b.material = m.material;
    b.xform = m.xform;
    if (m.uvs) {
        for (int c = 0; c < 3; c++) {
            b.uv[2 * c] = m.uvs[2 * (size_t)ti[c]];
            b.uv[2 * c + 1] = m.uvs[2 * (size_t)ti[c] + 1];
        }
    } else {  // triangle.h:24-26
        b.uv[0] = 0.0f; b.uv[1] = 0.0f; b.uv[2] = 1.0f; b.uv[3] = 0.0f; b.uv[4] = 0.0f; b.uv[5] = 1.0f;
    }
    return b;
}

// Conservative FP32 bounds of a baked primitive: (float) rounds to nearest, so every corner is
// stepped one ulp outward.
RT_HD inline void prim_bounds(const BakedPrim& b, float lo[3], float hi[3]) {
    const float big = 3.402823466e+38f;
    for (int k = 0; k < 3; k++) { lo[k] = big; hi[k] = -big; }
    auto grow = [&](D3 p, double pad) {
        const double c[3] = {p.x, p.y, p.z};
        for (int k = 0; k < 3; k++) {
            float l = nextafterf((float)dsub(c[k], pad), -INFINITY), h = nextafterf((float)dadd(c[k], pad), INFINITY);
            lo[k] = l < lo[k] ? l : lo[k];
            hi[k] = h > hi[k] ? h : hi[k];
        }
    };
    if (b.dev_type == PREP_SPHERE) {
        grow(b.a, b.radius);
    } else if (b.dev_type == PREP_MSPHERE) {
        grow(b.a, b.radius);
        grow(b.a + b.b, b.radius);
    } else if (b.dev_type == PREP_QUAD) {
        grow(b.a, 0); grow(b.a + b.b, 0); grow(b.a + b.c, 0); grow(b.a + b.b + b.c, 0);
    } else {
        grow(b.a, 0); grow(b.b, 0); grow(b.c, 0);
    }
}

// ---- device records (layout: DESIGN.md section 2) ------------------------------------------
struct F4 { float x, y, z, w; };
struct I4 { int x, y, z, w; };
RT_HD inline float int_bits_as_float(int v) {
    union { int i; float f; } u;
    u.i = v;
    return u.f;
}

struct SphereRec { F4 g; double d[4]; I4 sh; };
struct MSphereRec { F4 g0, g1; double d[8]; I4 sh; };
struct QuadRec { F4 q[3]; double d[12]; I4 sh; };
struct TriRec { F4 t[3]; double d[9]; F4 sh[3]; };

RT_HD inline SphereRec make_sphere(const BakedPrim& b) {
    SphereRec r;
    r.g = F4{(float)b.a.x, (float)b.a.y, (float)b.a.z, (float)b.radius};
    r.d[0] = b.a.x; r.d[1] = b.a.y; r.d[2] = b.a.z; r.d[3] = b.radius;
    r.sh = I4{b.material, b.xform, b.prim_id, 0};
    return r;
}
RT_HD inline MSphereRec make_msphere(const BakedPrim& b) {
    MSphereRec r;
    r.g0 = F4{(float)b.a.x, (float)b.a.y, (float)b.a.z, (float)b.radius};
    r.g1 = F4{(float)b.b.x, (float)b.b.y, (float)b.b.z, 0.0f};
    r.d[0] = b.a.x; r.d[1] = b.a.y; r.d[2] = b.a.z; r.d[3] = b.radius;
    r.d[4] = b.b.x; r.d[5] = b.b.y; r.d[6] = b.b.z; r.d[7] = 0.0;
    r.sh = I4{b.material, b.xform, b.prim_id, 0};
    return r;
}
// quad.h:13-21: n = u x v, normal = unit(n), D = normal.Q, w = n / (n.n);
// alpha = w.(p x v) = A.(P - Q) with A = v x w, beta = w.(u x p) = B.(P - Q) with B = w x u
RT_HD inline QuadRec make_quad(const BakedPrim& b) {
    QuadRec r;
    D3 n = dcross(b.b, b.c);
    D3 normal = dunit(n);
    double D = ddot(normal, b.a);
    D3 w = (1.0 / ddot(n, n)) * n;
    D3 A = dcross(b.c, w), B = dcross(w, b.b);
    double a0 = ddot(A, b.a), b0 = ddot(B, b.a);
    r.q[0] = F4{(float)normal.x, (float)normal.y, (float)normal.z, (float)D};
    r.q[1] = F4{(float)A.x, (float)A.y, (float)A.z, (float)a0};
    r.q[2] = F4{(float)B.x, (float)B.y, (float)B.z, (float)b0};
    const double d[12] = {normal.x, normal.y, normal.z, D, A.x, A.y, A.z, a0, B.x, B.y, B.z, b0};
    for (int k = 0; k < 12; k++) r.d[k] = d[k];
    r.sh = I4{b.material, 0, b.prim_id, 0};
    return r;
}
// triangle.h:21-22: normal = unit((p1 - p0) x (p2 - p0)); the edges are stored, not recomputed per ray
RT_HD inline TriRec make_triangle(const BakedPrim& b) {
    TriRec r;
    D3 e1 = b.b - b.a, e2 = b.c - b.a;
    D3 normal = dunit(dcross(e1, e2));
    r.t[0] = F4{(float)b.a.x, (float)b.a.y, (float)b.a.z, 0.0f};
    r.t[1] = F4{(float)e1.x, (float)e1.y, (float)e1.z, 0.0f};
    r.t[2] = F4{(float)e2.x, (float)e2.y, (float)e2.z, 0.0f};
    const double d[9] = {b.a.x, b.a.y, b.a.z, e1.x, e1.y, e1.z, e2.x, e2.y, e2.z};
    for (int k = 0; k < 9; k++) r.d[k] = d[k];
    r.sh[0] = F4{(float)normal.x, (float)normal.y, (float)normal.z, int_bits_as_float(b.material)};
    r.sh[1] = F4{b.uv[0], b.uv[1], b.uv[2], b.uv[3]};
    r.sh[2] = F4{b.uv[4], b.uv[5], int_bits_as_float(b.prim_id), 0.0f};
    return r;
}

// conservative outward padding of a node's child box (the FP32 slab test must never cull a true hit)
RT_HD inline void pad_box(const float lo[3], const float hi[3], float out_lo[3], float out_hi[3]) {
    const float pad = 1e-6f;
    for (int k = 0; k < 3; k++) {
        float m = fabsf(lo[k]) > fabsf(hi[k]) ? fabsf(lo[k]) : fabsf(hi[k]);
        float e = pad * (m > 1.0f ? m : 1.0f);
        out_lo[k] = lo[k] - e;
        out_hi[k] = hi[k] + e;
    }
}

// leaf link of the 64-byte node: ~(type << 28 | (count - 1) << 25 | first)
RT_HD inline int32_t leaf_link(uint32_t type, uint32_t count, uint32_t first) {
    return (int32_t) ~((type << 28) | ((count - 1u) << 25) | first);
}

}  // namespace rtprep
