// rtow_host.h — host-side mirror of the reference's scene-construction API.
//
// A program written against the reference (main.cpp:1-13 includes, main.cpp:128-471
// scene code) keeps compiling against this header set: the same class names and
// constructor signatures (sphere, quad, box(), triangle, triangle_quad, mesh::loadObj,
// translate, rotate_y, constant_medium, bvh_node, hittable_list, the materials, the
// textures, point_light, camera with the public fields of Camera.txt:39-52).
//
// What is different: none of these classes can intersect or shade anything.  They only
// record what was constructed and know how to FLATTEN themselves into the POD arrays of
// include/rt_b200.h; camera::render() (same signature as Camera.txt:54) flattens the
// world once and hands it to the CUDA library (rt_upload_scene / rt_render /
// rt_download).  There is no CPU rendering path in this header.
//
// The forwarding headers next to this file (sphere.h, quad.h, camera.h, glm.hpp, ...)
// exist so that the reference's #include lines resolve.
#ifndef RTB200_RTOW_HOST_H
#define RTB200_RTOW_HOST_H

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <limits>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "frame_io.h"
#include "host_rng.h"
#include "rt_b200.h"

// ---------------------------------------------------------------------------
// rtweekend.h
// ---------------------------------------------------------------------------
using std::make_shared;
using std::shared_ptr;

const double infinity = std::numeric_limits<double>::infinity();
const double pi = 3.1415926535897932385;

inline double degrees_to_radians(double degrees) { return degrees * pi / 180.0; }

// rtweekend.h:26-36 with rand() replaced by the thread-local generator (host_rng.h).
inline double random_double() { return rtb200::host_rand31() / 2147483648.0; }
inline double random_double(double lo, double hi) { return lo + (hi - lo) * random_double(); }
inline int random_int(int lo, int hi) { return int(random_double(lo, hi + 1)); }

// ---------------------------------------------------------------------------
// vec3.h / ray.h / interval.h / aabb.h — value types used by scene code
// ---------------------------------------------------------------------------
class vec3 {
  public:
    double e[3];
    vec3() : e{0, 0, 0} {}
    vec3(double a, double b, double c) : e{a, b, c} {}
    double x() const { return e[0]; }
    double y() const { return e[1]; }
    double z() const { return e[2]; }
    vec3 operator-() const { return vec3(-e[0], -e[1], -e[2]); }
    double operator[](int i) const { return e[i]; }
    double& operator[](int i) { return e[i]; }
    vec3& operator+=(const vec3& o) { e[0] += o.e[0]; e[1] += o.e[1]; e[2] += o.e[2]; return *this; }
    vec3& operator*=(double s) { e[0] *= s; e[1] *= s; e[2] *= s; return *this; }
    vec3& operator/=(double s) { return *this *= 1 / s; }
    bool operator==(const vec3& o) const { return e[0] == o.e[0] && e[1] == o.e[1] && e[2] == o.e[2]; }
    double length_squared() const { return e[0] * e[0] + e[1] * e[1] + e[2] * e[2]; }
    double length() const { return std::sqrt(length_squared()); }
    bool near_zero() const {
        const double s = 1e-8;
        return std::fabs(e[0]) < s && std::fabs(e[1]) < s && std::fabs(e[2]) < s;
    }
    // vec3.h:50-56 writes `vec3(random_double(), random_double(), random_double())`;
    // argument evaluation order is unspecified in C++ and g++ (the compiler the oracle is
    // built with) evaluates right to left, so the FIRST draw lands in z.  Sequenced
    // explicitly here so that scenes and Perlin tables match the oracle's
    // (checked by tests/test_scenes.py against the compiled reference).
    static vec3 random() {
        double c = random_double(), b = random_double(), a = random_double();
        return vec3(a, b, c);
    }
    static vec3 random(double lo, double hi) {
        double c = random_double(lo, hi), b = random_double(lo, hi), a = random_double(lo, hi);
        return vec3(a, b, c);
    }
};
using point3 = vec3;
using color = vec3;

inline std::ostream& operator<<(std::ostream& out, const vec3& v) { return out << v.e[0] << ' ' << v.e[1] << ' ' << v.e[2]; }
inline vec3 operator+(const vec3& a, const vec3& b) { return vec3(a.e[0] + b.e[0], a.e[1] + b.e[1], a.e[2] + b.e[2]); }
inline vec3 operator-(const vec3& a, const vec3& b) { return vec3(a.e[0] - b.e[0], a.e[1] - b.e[1], a.e[2] - b.e[2]); }
inline vec3 operator*(const vec3& a, const vec3& b) { return vec3(a.e[0] * b.e[0], a.e[1] * b.e[1], a.e[2] * b.e[2]); }
inline vec3 operator*(double s, const vec3& v) { return vec3(s * v.e[0], s * v.e[1], s * v.e[2]); }
inline vec3 operator*(const vec3& v, double s) { return s * v; }
inline vec3 operator/(const vec3& v, double s) { return (1 / s) * v; }
inline double dot(const vec3& a, const vec3& b) { return a.e[0] * b.e[0] + a.e[1] * b.e[1] + a.e[2] * b.e[2]; }
inline vec3 cross(const vec3& a, const vec3& b) {
    return vec3(a.e[1] * b.e[2] - a.e[2] * b.e[1], a.e[2] * b.e[0] - a.e[0] * b.e[2], a.e[0] * b.e[1] - a.e[1] * b.e[0]);
}
inline vec3 unit_vector(const vec3& v) { return v / v.length(); }

class ray {
  public:
    ray() {}
    ray(const point3& o, const vec3& d, double time) : orig(o), dir(d), tm(time) {}
    ray(const point3& o, const vec3& d) : ray(o, d, 0) {}
    const point3& origin() const { return orig; }
    const vec3& direction() const { return dir; }
    double time() const { return tm; }
    point3 at(double t) const { return orig + t * dir; }
  private:
    point3 orig;
    vec3 dir;
    double tm = 0;
};

class interval {
  public:
    double min, max;
    interval() : min(+infinity), max(-infinity) {}
    interval(double lo, double hi) : min(lo), max(hi) {}
    interval(const interval& a, const interval& b) {
        min = a.min <= b.min ? a.min : b.min;
        max = a.max >= b.max ? a.max : b.max;
    }
    double size() const { return max - min; }
    bool contains(double x) const { return min <= x && x <= max; }
    bool surrounds(double x) const { return min < x && x < max; }
    double clamp(double x) const { return x < min ? min : (x > max ? max : x); }
    interval expand(double delta) const { return interval(min - delta / 2, max + delta / 2); }
    static interval empty() { return interval(+infinity, -infinity); }
    static interval universe() { return interval(-infinity, +infinity); }
};
inline interval operator+(const interval& iv, double d) { return interval(iv.min + d, iv.max + d); }
inline interval operator+(double d, const interval& iv) { return iv + d; }

// Bounding boxes are only used on the host to replay the reference's BVH ordering
// (bvh.h:24-44), so their values follow aabb.h bit for bit: the two-point form does
// not pad (aabb.h:21-45), the interval and merge forms do (aabb.h:16-19, 47-53).
class aabb {
  public:
    interval x, y, z;
    aabb() {}
    aabb(const interval& ix, const interval& iy, const interval& iz) : x(ix), y(iy), z(iz) { pad(); }
    aabb(const point3& a, const point3& b) {
        x = a[0] <= b[0] ? interval(a[0], b[0]) : interval(b[0], a[0]);
        y = a[1] <= b[1] ? interval(a[1], b[1]) : interval(b[1], a[1]);
        z = a[2] <= b[2] ? interval(a[2], b[2]) : interval(b[2], a[2]);
    }
    aabb(const aabb& a, const aabb& b) : x(a.x, b.x), y(a.y, b.y), z(a.z, b.z) { pad(); }
    const interval& axis_interval(int n) const { return n == 1 ? y : (n == 2 ? z : x); }
    int longest_axis() const {
        if (x.size() > y.size()) return x.size() > z.size() ? 0 : 2;
        return y.size() > z.size() ? 1 : 2;
    }
    static aabb empty() { return aabb(interval::empty(), interval::empty(), interval::empty()); }
  private:
    void pad() {
        const double delta = 0.0001;
        if (x.size() < delta) x = x.expand(delta);
        if (y.size() < delta) y = y.expand(delta);
        if (z.size() < delta) z = z.expand(delta);
    }
};
inline aabb operator+(const aabb& b, const vec3& o) { return aabb(b.x + o.x(), b.y + o.y(), b.z + o.z()); }
inline aabb operator+(const vec3& o, const aabb& b) { return b + o; }

// ---------------------------------------------------------------------------
// a small glm-compatible subset (the reference vendors GLM 0.9.8.5 only for
// glm::vec2 UVs in triangle.h and glm::mat4 vertex transforms in mesh.h).  If the
// real GLM has already been included this block is skipped.
// ---------------------------------------------------------------------------
#ifndef GLM_VERSION
#define RTB200_GLM_COMPAT 1
namespace glm {
struct vec2 {
    float x, y;
    vec2() : x(0), y(0) {}
    vec2(float a, float b) : x(a), y(b) {}
};
struct vec3 {
    float x, y, z;
    vec3() : x(0), y(0), z(0) {}
    explicit vec3(float s) : x(s), y(s), z(s) {}
    vec3(float a, float b, float c) : x(a), y(b), z(c) {}
    float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
};
struct vec4 {
    float x, y, z, w;
    vec4() : x(0), y(0), z(0), w(0) {}
    vec4(float a, float b, float c, float d) : x(a), y(b), z(c), w(d) {}
    vec4(const vec3& v, float d) : x(v.x), y(v.y), z(v.z), w(d) {}
    float operator[](int i) const { return i == 0 ? x : (i == 1 ? y : (i == 2 ? z : w)); }
};
inline vec4 operator*(const vec4& a, float s) { return vec4(a.x * s, a.y * s, a.z * s, a.w * s); }
inline vec4 operator+(const vec4& a, const vec4& b) { return vec4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
struct mat4 {
    vec4 c[4];  // column-major like GLM
    mat4() {}
    explicit mat4(float d) {
        c[0] = vec4(d, 0, 0, 0); c[1] = vec4(0, d, 0, 0); c[2] = vec4(0, 0, d, 0); c[3] = vec4(0, 0, 0, d);
    }
    vec4& operator[](int i) { return c[i]; }
    const vec4& operator[](int i) const { return c[i]; }
};
// same association as GLM's type_mat4x4.inl:526-537: (m0*v0 + m1*v1) + (m2*v2 + m3*v3)
inline vec4 operator*(const mat4& m, const vec4& v) {
    vec4 a0 = m[0] * v.x + m[1] * v.y;
    vec4 a1 = m[2] * v.z + m[3] * v.w;
    return a0 + a1;
}
inline float radians(float deg) { return deg * 0.01745329251994329576923690768489f; }
inline mat4 translate(const mat4& m, const vec3& v) {
    mat4 r(m);
    r[3] = m[0] * v.x + m[1] * v.y + m[2] * v.z + m[3];
    return r;
}
inline mat4 scale(const mat4& m, const vec3& v) {
    mat4 r;
    r[0] = m[0] * v.x; r[1] = m[1] * v.y; r[2] = m[2] * v.z; r[3] = m[3];
    return r;
}
inline mat4 rotate(const mat4& m, float angle, const vec3& axis_in) {
    const float c = std::cos(angle), s = std::sin(angle);
    const float inv = 1.0f / std::sqrt(axis_in.x * axis_in.x + axis_in.y * axis_in.y + axis_in.z * axis_in.z);
    const vec3 a(axis_in.x * inv, axis_in.y * inv, axis_in.z * inv);
    const vec3 t((1.0f - c) * a.x, (1.0f - c) * a.y, (1.0f - c) * a.z);
    float r00 = c + t.x * a.x, r01 = t.x * a.y + s * a.z, r02 = t.x * a.z - s * a.y;
    float r10 = t.y * a.x - s * a.z, r11 = c + t.y * a.y, r12 = t.y * a.z + s * a.x;
    float r20 = t.z * a.x + s * a.y, r21 = t.z * a.y - s * a.x, r22 = c + t.z * a.z;
    mat4 r;
    r[0] = m[0] * r00 + m[1] * r01 + m[2] * r02;
    r[1] = m[0] * r10 + m[1] * r11 + m[2] * r12;
    r[2] = m[0] * r20 + m[1] * r21 + m[2] * r22;
    r[3] = m[3];
    return r;
}
}  // namespace glm
#endif

// ---------------------------------------------------------------------------
// flattening machinery
// ---------------------------------------------------------------------------
class material;
class texture;
class hittable;

namespace rtb200 {

// std::vector whose resize() leaves trivially-constructible elements uninitialised: the big
// record arrays (a million triangles = 104 MB) are then first touched by the threads that fill them.
template <class T>
struct default_init_allocator : std::allocator<T> {
    template <class U> struct rebind { using other = default_init_allocator<U>; };
    using std::allocator<T>::allocator;
    template <class U> void construct(U* p) noexcept(std::is_nothrow_default_constructible<U>::value) { ::new (static_cast<void*>(p)) U; }
    template <class U, class... A> void construct(U* p, A&&... a) { ::new (static_cast<void*>(p)) U(std::forward<A>(a)...); }
};
template <class T> using pod_vector = std::vector<T, default_init_allocator<T>>;

// runs fn(part, n_parts) on up to 16 host threads (one part per thread; part 0 on the caller)
template <class F>
inline void parallel_parts(size_t n_parts, F&& fn) {
    std::vector<std::thread> pool;
    for (size_t i = 1; i < n_parts; i++) pool.emplace_back([&fn, i, n_parts] { fn(i, n_parts); });
    fn((size_t)0, n_parts);
    for (auto& t : pool) t.join();
}
// a whole file, read-only: mapped, not copied
class mapped_file {
  public:
    explicit mapped_file(const char* path) {
        fd = ::open(path, O_RDONLY);
        if (fd < 0) return;
        struct stat st;
        if (::fstat(fd, &st) != 0) { ::close(fd); fd = -1; return; }
        len = (size_t)st.st_size;
        if (len == 0) return;
        void* m = ::mmap(nullptr, len, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) { ::close(fd); fd = -1; len = 0; return; }
        ptr = (const char*)m;
    }
    ~mapped_file() {
        if (ptr) ::munmap((void*)ptr, len);
        if (fd >= 0) ::close(fd);
    }
    mapped_file(const mapped_file&) = delete;
    mapped_file& operator=(const mapped_file&) = delete;
    bool ok() const { return fd >= 0; }
    const char* data() const { return ptr ? ptr : ""; }
    size_t size() const { return len; }
  private:
    int fd = -1;
    const char* ptr = nullptr;
    size_t len = 0;
};

inline size_t host_parts(size_t work_items, size_t min_per_part) {
    const size_t hw = std::max(1u, std::thread::hardware_concurrency());
    return std::max<size_t>(1, std::min<size_t>({hw, (size_t)16, work_items / std::max<size_t>(1, min_per_part)}));
}

struct xform3 {
    double r[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    double t[3] = {0, 0, 0};
};

// The arrays of one indexed triangle mesh (rt_mesh), shared by the hittable that holds them and the
// flattened scenes that point at them.
struct mesh_arrays {
    pod_vector<float> positions;      // 3 per vertex
    pod_vector<uint32_t> indices;     // 3 per triangle
    pod_vector<float> uvs;            // 2 per texture coordinate; empty: every triangle gets (0,0), (1,0), (0,1)
    pod_vector<uint32_t> uv_indices;  // 3 per triangle; empty: the position indices
    size_t triangles() const { return indices.size() / 3; }
    // corner c of triangle k, widened to double (what an rt_triangle of the same face holds)
    void corner(size_t k, int c, double out[3]) const {
        const float* p = positions.data() + 3 * (size_t)indices[3 * k + c];
        for (int d = 0; d < 3; d++) out[d] = p[d];
    }
};

// Owns the POD arrays of one flattened scene and hands out an rt_scene_desc view.
struct flat_scene {
    pod_vector<rt_prim_ref> world, boundary_refs;
    std::vector<rt_sphere> spheres;
    std::vector<rt_quad> quads;
    pod_vector<rt_triangle> triangles;
    std::vector<rt_medium> media;
    std::vector<rt_xform> xforms;
    std::vector<rt_material> materials;
    std::vector<rt_texture> textures;
    std::vector<rt_image> images;
    std::vector<std::vector<uint8_t>> image_bytes;
    std::vector<rt_perlin> perlins;
    std::vector<rt_point_light> lights;
    std::vector<rt_mesh> meshes;
    std::vector<std::shared_ptr<const mesh_arrays>> mesh_data;  // keeps the arrays behind `meshes` alive (not copied)
    rt_camera camera{};

    rt_scene_desc desc() const {
        rt_scene_desc d;
        std::memset(&d, 0, sizeof d);
        d.struct_size = sizeof d;
        d.abi_version = RT_B200_ABI_VERSION;
        d.world = world.data();            d.n_world = (int32_t)world.size();
        d.boundary_refs = boundary_refs.data(); d.n_boundary_refs = (int32_t)boundary_refs.size();
        d.spheres = spheres.data();        d.n_spheres = (int32_t)spheres.size();
        d.quads = quads.data();            d.n_quads = (int32_t)quads.size();
        d.triangles = triangles.data();    d.n_triangles = (int32_t)triangles.size();
        d.media = media.data();            d.n_media = (int32_t)media.size();
        d.xforms = xforms.data();          d.n_xforms = (int32_t)xforms.size();
        d.materials = materials.data();    d.n_materials = (int32_t)materials.size();
        d.textures = textures.data();      d.n_textures = (int32_t)textures.size();
        d.images = images.data();          d.n_images = (int32_t)images.size();
        d.perlins = perlins.data();        d.n_perlins = (int32_t)perlins.size();
        d.lights = lights.data();          d.n_lights = (int32_t)lights.size();
        d.meshes = meshes.data();          d.n_meshes = (int32_t)meshes.size();
        d.camera = camera;
        return d;
    }

    // Identity of the flattened scene for checkpoint files (the ABI structs have no padding bytes).
    uint64_t hash() const {
        uint64_t h = 1469598103934665603ull;
        auto add = [&](const void* p, size_t n) { if (n) h = fnv1a(p, n, h); };
        add(world.data(), world.size() * sizeof(rt_prim_ref));
        add(boundary_refs.data(), boundary_refs.size() * sizeof(rt_prim_ref));
        add(spheres.data(), spheres.size() * sizeof(rt_sphere));
        add(quads.data(), quads.size() * sizeof(rt_quad));
        add(triangles.data(), triangles.size() * sizeof(rt_triangle));
        add(media.data(), media.size() * sizeof(rt_medium));
        add(xforms.data(), xforms.size() * sizeof(rt_xform));
        add(materials.data(), materials.size() * sizeof(rt_material));
        add(textures.data(), textures.size() * sizeof(rt_texture));
        for (size_t i = 0; i < images.size(); i++) {
            add(&images[i].width, sizeof(int32_t));
            add(&images[i].height, sizeof(int32_t));
            add(images[i].rgb, (size_t)images[i].width * images[i].height * 3);
        }
        add(perlins.data(), perlins.size() * sizeof(rt_perlin));
        add(lights.data(), lights.size() * sizeof(rt_point_light));
        for (const rt_mesh& m : meshes) {
            const int32_t f[6] = {m.n_vertices, m.n_triangles, m.n_uvs, m.material, m.xform, (m.uvs ? 1 : 0) | (m.uv_indices ? 2 : 0)};
            add(f, sizeof f);
            add(m.positions, (size_t)m.n_vertices * 3 * sizeof(float));
            add(m.indices, (size_t)m.n_triangles * 3 * sizeof(uint32_t));
            if (m.uvs) add(m.uvs, (size_t)m.n_uvs * 2 * sizeof(float));
            if (m.uv_indices) add(m.uv_indices, (size_t)m.n_triangles * 3 * sizeof(uint32_t));
        }
        add(&camera, sizeof camera);
        return h;
    }
};

// The visitor every hittable / material / texture flattens itself into.
class flattener {
  public:
    explicit flattener(flat_scene& out) : fs(out) { stack.push_back({xform3(), -1}); }

    // --- instance transforms (hittable.h:39-65 translate, :67-146 rotate_y) -------
    void push_translate(const vec3& off) {
        xform3 x;
        x.t[0] = off.x(); x.t[1] = off.y(); x.t[2] = off.z();
        push(x);
    }
    void push_rotate_y(double sin_t, double cos_t) {
        // world = (c*x + s*z, y, -s*x + c*z)   (hittable.h:121-125)
        xform3 x;
        x.r[0] = cos_t; x.r[2] = sin_t; x.r[6] = -sin_t; x.r[8] = cos_t;
        push(x);
    }
    void pop() { stack.pop_back(); }

    int current_xform() {
        entry& top = stack.back();
        if (stack.size() == 1) return -1;
        if (top.index < 0) {
            rt_xform x;
            std::memcpy(x.r, top.x.r, sizeof x.r);
            std::memcpy(x.t, top.x.t, sizeof x.t);
            fs.xforms.push_back(x);
            top.index = (int)fs.xforms.size() - 1;
        }
        return top.index;
    }

    // --- leaves ---------------------------------------------------------------------
    void add_sphere(const vec3& c0, const vec3& cvec, double radius, const shared_ptr<material>& m) {
        rt_sphere s;
        std::memset(&s, 0, sizeof s);
        for (int k = 0; k < 3; k++) { s.center0[k] = c0[k]; s.center_vec[k] = cvec[k]; }
        s.radius = radius;
        s.material = boundary_depth > 0 ? -1 : material_id(m);
        s.xform = current_xform();
        fs.spheres.push_back(s);
        add_ref(RT_PRIM_SPHERE, (int)fs.spheres.size() - 1);
    }
    void add_quad(const vec3& Q, const vec3& u, const vec3& v, const shared_ptr<material>& m) {
        rt_quad q;
        std::memset(&q, 0, sizeof q);
        for (int k = 0; k < 3; k++) { q.Q[k] = Q[k]; q.u[k] = u[k]; q.v[k] = v[k]; }
        q.material = boundary_depth > 0 ? -1 : material_id(m);
        q.xform = current_xform();
        fs.quads.push_back(q);
        add_ref(RT_PRIM_QUAD, (int)fs.quads.size() - 1);
    }
    void add_triangle(const vec3& p0, const vec3& p1, const vec3& p2, const float uv[6], const shared_ptr<material>& m) {
        rt_triangle t;
        std::memset(&t, 0, sizeof t);
        for (int k = 0; k < 3; k++) { t.p0[k] = p0[k]; t.p1[k] = p1[k]; t.p2[k] = p2[k]; }
        t.uv0[0] = uv[0]; t.uv0[1] = uv[1]; t.uv1[0] = uv[2]; t.uv1[1] = uv[3]; t.uv2[0] = uv[4]; t.uv2[1] = uv[5];
        t.material = boundary_depth > 0 ? -1 : material_id(m);
        t.xform = current_xform();
        fs.triangles.push_back(t);
        add_ref(RT_PRIM_TRIANGLE, (int)fs.triangles.size() - 1);
    }

    // Bulk version for triangle_soup: `tris` already holds ABI records (positions, uvs); only the
    // material and transform indices are resolved here.  One material lookup, one append.
    void add_triangles(const pod_vector<rt_triangle>& tris, const shared_ptr<material>& m) {
        if (tris.empty()) return;
        const int mat = boundary_depth > 0 ? -1 : material_id(m);
        const int xf = current_xform();
        const size_t first = fs.triangles.size(), n = tris.size();
        fs.triangles.resize(first + n);
        pod_vector<rt_prim_ref>& refs = boundary_depth > 0 ? fs.boundary_refs : fs.world;
        const size_t r0 = refs.size();
        refs.resize(r0 + n);
        rt_triangle* dst = fs.triangles.data() + first;
        rt_prim_ref* ref = refs.data() + r0;
        parallel_parts(host_parts(n, 1 << 15), [&](size_t part, size_t parts) {
            const size_t a = n * part / parts, b = n * (part + 1) / parts;
            std::memcpy(dst + a, tris.data() + a, (b - a) * sizeof(rt_triangle));
            for (size_t i = a; i < b; i++) {
                dst[i].material = mat;
                dst[i].xform = xf;
                ref[i] = rt_prim_ref{RT_PRIM_TRIANGLE, (int32_t)(first + i)};
            }
        });
    }

    // An indexed mesh: one rt_mesh and ONE world ref (its triangles take consecutive canonical ids, as a soup's
    // would).  Inside a medium boundary, where meshes are not accepted, it becomes that many rt_triangles.
    void add_mesh(const std::shared_ptr<const mesh_arrays>& a, const shared_ptr<material>& m) {
        const size_t n = a->triangles();
        if (n == 0) return;
        if (boundary_depth > 0) {
            pod_vector<rt_triangle> tris(n);
            for (size_t k = 0; k < n; k++) {
                rt_triangle& t = tris[k];
                std::memset(&t, 0, sizeof t);
                a->corner(k, 0, t.p0); a->corner(k, 1, t.p1); a->corner(k, 2, t.p2);
                float* uv[3] = {t.uv0, t.uv1, t.uv2};
                for (int c = 0; c < 3; c++) {
                    if (a->uvs.empty()) {  // triangle.h:24-26
                        uv[c][0] = c == 1 ? 1.0f : 0.0f;
                        uv[c][1] = c == 2 ? 1.0f : 0.0f;
                    } else {
                        const uint32_t i = (a->uv_indices.empty() ? a->indices : a->uv_indices)[3 * k + c];
                        uv[c][0] = a->uvs[2 * (size_t)i];
                        uv[c][1] = a->uvs[2 * (size_t)i + 1];
                    }
                }
            }
            add_triangles(tris, m);
            return;
        }
        rt_mesh r;
        std::memset(&r, 0, sizeof r);
        r.positions = a->positions.data();
        r.indices = a->indices.data();
        r.uvs = a->uvs.empty() ? nullptr : a->uvs.data();
        r.uv_indices = a->uv_indices.empty() ? nullptr : a->uv_indices.data();
        r.n_vertices = (int32_t)(a->positions.size() / 3);
        r.n_triangles = (int32_t)n;
        r.n_uvs = (int32_t)(a->uvs.size() / 2);
        r.material = material_id(m);
        r.xform = current_xform();
        fs.meshes.push_back(r);
        fs.mesh_data.push_back(a);
        add_ref(RT_PRIM_MESH, (int)fs.meshes.size() - 1);
    }

    // --- participating media (constant_medium.h:8-61) -------------------------------
    void add_medium(const hittable& boundary, double density, const shared_ptr<material>& phase);

    // --- BVH leaf multiplicity (bvh.h:31-33, SURVEY Q15) ---------------------------
    int multiplicity = 1;

    int material_id(const shared_ptr<material>& m);
    int texture_id(const shared_ptr<texture>& t);

    flat_scene& fs;

  private:
    struct entry { xform3 x; int index; };
    std::vector<entry> stack;
    int boundary_depth = 0;
    std::map<const material*, int> mat_ids;
    std::map<const texture*, int> tex_ids;

    void push(const xform3& local) {
        // world = Rp * (Rl * p + tl) + tp
        const xform3& p = stack.back().x;
        xform3 c;
        for (int i = 0; i < 3; i++) {
            for (int j = 0; j < 3; j++) {
                double acc = 0;
                for (int k = 0; k < 3; k++) acc += p.r[i * 3 + k] * local.r[k * 3 + j];
                c.r[i * 3 + j] = acc;
            }
            double acc = p.t[i];
            for (int k = 0; k < 3; k++) acc += p.r[i * 3 + k] * local.t[k];
            c.t[i] = acc;
        }
        stack.push_back({c, -1});
    }
    void add_ref(int type, int index) {
        rt_prim_ref r{type, index};
        (boundary_depth > 0 ? fs.boundary_refs : fs.world).push_back(r);
    }
};

}  // namespace rtb200

// ---------------------------------------------------------------------------
// perlin.h / rtw_stb_image.h / texture.h
// ---------------------------------------------------------------------------
// Draws exactly the random numbers perlin.h:6-13,58-71 draws, in the same order, so
// that the tables match the oracle's when both start from the same seed: 256 x
// unit_vector(vec3::random(-1,1)), then three permutations whose swap target is
// random_int(0,1) (the reference's weak shuffle, SURVEY Q2 — kept on purpose).
class perlin {
  public:
    perlin() {
        for (int i = 0; i < point_count; i++) randVec[i] = unit_vector(vec3::random(-1, 1));
        make_perm(perm_x);
        make_perm(perm_y);
        make_perm(perm_z);
    }
    void export_tables(rt_perlin& out) const {
        for (int i = 0; i < point_count; i++) {
            for (int k = 0; k < 3; k++) out.randvec[i][k] = randVec[i][k];
            out.perm_x[i] = perm_x[i]; out.perm_y[i] = perm_y[i]; out.perm_z[i] = perm_z[i];
        }
    }
  private:
    static const int point_count = 256;
    vec3 randVec[point_count];
    int perm_x[point_count], perm_y[point_count], perm_z[point_count];
    static void make_perm(int* p) {
        for (int i = 0; i < point_count; i++) p[i] = i;
        for (int i = point_count - 1; i > 0; i--) {
            int target = random_int(0, 1);
            std::swap(p[i], p[target]);
        }
    }
};

// Image loader.  The reference decodes with the vendored stb_image (out of the hot
// path's scope); what the hot path consumes is rtw_image::bdata — RGB bytes that went
// through stbi_loadf's gamma-2.2 linearisation (stb_image.h:1869) and
// float_to_byte (rtw_stb_image.h:99-105).  This mirror reads binary PPM/PGM (P6/P5)
// natively and applies the same byte -> float -> byte mapping; define
// RTB200_USE_STB_IMAGE (with stb_image.h on the include path) to decode JPEG/PNG the
// way the reference does.
class rtw_image {
  public:
    rtw_image() {}
    rtw_image(const char* image_filename) {
        std::string filename(image_filename);
        const char* imagedir = std::getenv("RTW_IMAGES");
        if (imagedir && load(std::string(imagedir) + "/" + filename)) return;
        if (load(filename)) return;
        std::string prefix = "images/";
        for (int up = 0; up < 7; up++) {  // images/, ../images/, ... six levels up (rtw_stb_image.h:35-43)
            if (load(prefix + filename)) return;
            prefix = "../" + prefix;
        }
        std::cerr << "ERROR: Could not load image file '" << image_filename << "'.\n";
    }
    // construct from raw 8-bit sRGB-ish texels (what a decoder would hand to ldr_to_hdr)
    rtw_image(int w, int h, const uint8_t* rgb_in) { assign(w, h, rgb_in); }

    bool load(const std::string& filename) {
#ifdef RTB200_USE_STB_IMAGE
        int n = 3, w = 0, h = 0;
        unsigned char* raw = stbi_load(filename.c_str(), &w, &h, &n, 3);
        if (!raw) return false;
        assign(w, h, raw);
        stbi_image_free(raw);
        return true;
#else
        std::ifstream f(filename, std::ios::binary);
        if (!f.is_open()) return false;
        std::string magic;
        f >> magic;
        if (magic != "P6" && magic != "P5") return false;
        int vals[3], got = 0;
        while (got < 3) {  // width height maxval, '#' comments allowed
            int ch = f.peek();
            if (ch == '#') { std::string skip; std::getline(f, skip); continue; }
            if (std::isspace(ch)) { f.get(); continue; }
            if (!(f >> vals[got])) return false;
            got++;
        }
        f.get();  // the single whitespace byte after maxval
        if (vals[0] <= 0 || vals[1] <= 0 || vals[2] != 255) return false;
        const int comps = magic == "P6" ? 3 : 1;
        std::vector<uint8_t> raw((size_t)vals[0] * vals[1] * comps);
        f.read((char*)raw.data(), (std::streamsize)raw.size());
        if ((size_t)f.gcount() != raw.size()) return false;
        if (comps == 1) {
            std::vector<uint8_t> rgb3((size_t)vals[0] * vals[1] * 3);
            for (size_t i = 0; i < raw.size(); i++) rgb3[3 * i] = rgb3[3 * i + 1] = rgb3[3 * i + 2] = raw[i];
            assign(vals[0], vals[1], rgb3.data());
        } else {
            assign(vals[0], vals[1], raw.data());
        }
        return true;
#endif
    }
    int width() const { return bdata.empty() ? 0 : image_width; }
    int height() const { return bdata.empty() ? 0 : image_height; }
    const std::vector<uint8_t>& bytes() const { return bdata; }

  private:
    int image_width = 0, image_height = 0;
    std::vector<uint8_t> bdata;  // linear 8-bit texels, 3 per pixel, top row first

    void assign(int w, int h, const uint8_t* rgb_in) {
        // 256-entry table of  float_to_byte((float)pow(b/255.0f, 2.2f))
        uint8_t lut[256];
        for (int b = 0; b < 256; b++) {
            float lin = (float)(std::pow(b / 255.0f, 2.2f) * 1.0f);
            lut[b] = lin <= 0.0 ? 0 : (1.0 <= lin ? 255 : static_cast<unsigned char>(256.0 * lin));
        }
        image_width = w; image_height = h;
        bdata.resize((size_t)w * h * 3);
        for (size_t i = 0; i < bdata.size(); i++) bdata[i] = lut[rgb_in[i]];
    }
};

class texture {
  public:
    virtual ~texture() = default;
    virtual void describe(rtb200::flattener& f, rt_texture& out) const = 0;
};

class solid_color : public texture {
  public:
    solid_color(const color& c) : albedo(c) {}
    solid_color(double r, double g, double b) : albedo(r, g, b) {}
    void describe(rtb200::flattener&, rt_texture& out) const override {
        out.type = RT_TEX_SOLID;
        for (int k = 0; k < 3; k++) out.color[k] = albedo[k];
    }
  private:
    color albedo;
};

class checker_texture : public texture {  // texture.h:34-56
  public:
    checker_texture(double scale, shared_ptr<texture> e, shared_ptr<texture> o) : inv_scale(1.0 / scale), even(e), odd(o) {}
    checker_texture(double scale, const color& c1, const color& c2)
        : checker_texture(scale, make_shared<solid_color>(c1), make_shared<solid_color>(c2)) {}
    void describe(rtb200::flattener& f, rt_texture& out) const override {
        out.type = RT_TEX_CHECKER;
        out.scale = inv_scale;
        out.even = f.texture_id(even);
        out.odd = f.texture_id(odd);
    }
  private:
    double inv_scale;
    shared_ptr<texture> even, odd;
};

class checker_texture_triangle : public texture {  // texture.h:58-84 (UV space, fixed 10x10)
  public:
    checker_texture_triangle(double scale, shared_ptr<texture> e, shared_ptr<texture> o)
        : inv_scale(1.0 / std::max(0.01, scale)), even(e), odd(o) {}
    checker_texture_triangle(double scale, const color& c1, const color& c2)
        : checker_texture_triangle(scale, make_shared<solid_color>(c1), make_shared<solid_color>(c2)) {}
    void describe(rtb200::flattener& f, rt_texture& out) const override {
        out.type = RT_TEX_CHECKER_TRIANGLE;
        out.scale = inv_scale;
        out.even = f.texture_id(even);
        out.odd = f.texture_id(odd);
    }
  private:
    double inv_scale;
    shared_ptr<texture> even, odd;
};

class image_texture : public texture {  // texture.h:86-108
  public:
    image_texture(const char* filename) : image(filename) {}
    image_texture(int w, int h, const uint8_t* rgb_in) : image(w, h, rgb_in) {}
    void describe(rtb200::flattener& f, rt_texture& out) const override {
        out.type = RT_TEX_IMAGE;
        out.image = -1;
        if (image.width() > 0 && image.height() > 0) {
            f.fs.image_bytes.push_back(image.bytes());
            rt_image im;
            im.width = image.width(); im.height = image.height();
            im.rgb = nullptr;  // patched after flattening (vector storage may move)
            f.fs.images.push_back(im);
            out.image = (int)f.fs.images.size() - 1;
        }
    }
  private:
    rtw_image image;
};

class noise_texture : public texture {  // texture.h:110-120
  public:
    noise_texture(double s) : scale(s) {}
    void describe(rtb200::flattener& f, rt_texture& out) const override {
        out.type = RT_TEX_NOISE;
        out.scale = scale;
        rt_perlin p;
        noise.export_tables(p);
        f.fs.perlins.push_back(p);
        out.perlin = (int)f.fs.perlins.size() - 1;
    }
  private:
    perlin noise;
    double scale;
};

// ---------------------------------------------------------------------------
// material.h
// ---------------------------------------------------------------------------
class material {
  public:
    virtual ~material() = default;
    virtual void describe(rtb200::flattener& f, rt_material& out) const = 0;
};

class lambertian : public material {
  public:
    lambertian(const color& albedo) : tex(make_shared<solid_color>(albedo)) {}
    lambertian(shared_ptr<texture> t) : tex(t) {}
    void describe(rtb200::flattener& f, rt_material& out) const override {
        out.type = RT_MAT_LAMBERTIAN;
        out.texture = f.texture_id(tex);
    }
  private:
    shared_ptr<texture> tex;
};

class dielectric : public material {
  public:
    dielectric(double ri) : refraction_index(ri) {}
    void describe(rtb200::flattener&, rt_material& out) const override {
        out.type = RT_MAT_DIELECTRIC;
        out.param = refraction_index;
    }
  private:
    double refraction_index;
};

class metal : public material {
  public:
    metal(const color& a, double fz) : albedo(a), fuzz(fz < 1 ? fz : 1) {}
    void describe(rtb200::flattener&, rt_material& out) const override {
        out.type = RT_MAT_METAL;
        for (int k = 0; k < 3; k++) out.albedo[k] = albedo[k];
        out.param = fuzz;
    }
  private:
    color albedo;
    double fuzz;
};

class diffuse_light : public material {
  public:
    diffuse_light(shared_ptr<texture> t) : tex(t) {}
    diffuse_light(const color& emit) : tex(make_shared<solid_color>(emit)) {}
    void describe(rtb200::flattener& f, rt_material& out) const override {
        out.type = RT_MAT_DIFFUSE_LIGHT;
        out.texture = f.texture_id(tex);
    }
  private:
    shared_ptr<texture> tex;
};

class emissive_light : public material {
  public:
    emissive_light(shared_ptr<texture> t) : tex(t) {}
    emissive_light(const color& emit) : tex(make_shared<solid_color>(emit)) {}
    void describe(rtb200::flattener& f, rt_material& out) const override {
        out.type = RT_MAT_EMISSIVE_LIGHT;
        out.texture = f.texture_id(tex);
    }
  private:
    shared_ptr<texture> tex;
};

class isotropic : public material {
  public:
    isotropic(const color& albedo) : tex(make_shared<solid_color>(albedo)) {}
    isotropic(shared_ptr<texture> t) : tex(t) {}
    void describe(rtb200::flattener& f, rt_material& out) const override {
        out.type = RT_MAT_ISOTROPIC;
        out.texture = f.texture_id(tex);
    }
  private:
    shared_ptr<texture> tex;
};

class specular : public material {
  public:
    specular(const color& a, double sh) : albedo(a), shininess(sh) {}
    void describe(rtb200::flattener&, rt_material& out) const override {
        out.type = RT_MAT_SPECULAR;
        for (int k = 0; k < 3; k++) out.albedo[k] = albedo[k];
        out.param = shininess;
    }
  private:
    color albedo;
    double shininess;
};

inline int rtb200::flattener::texture_id(const shared_ptr<texture>& t) {
    if (!t) return -1;
    auto it = tex_ids.find(t.get());
    if (it != tex_ids.end()) return it->second;
    rt_texture rec;
    std::memset(&rec, 0, sizeof rec);
    rec.even = rec.odd = rec.image = rec.perlin = -1;
    int id = (int)fs.textures.size();
    fs.textures.push_back(rec);  // reserve the slot first: children get higher ids
    tex_ids[t.get()] = id;
    t->describe(*this, rec);
    fs.textures[id] = rec;
    return id;
}

inline int rtb200::flattener::material_id(const shared_ptr<material>& m) {
    if (!m) return -1;
    auto it = mat_ids.find(m.get());
    if (it != mat_ids.end()) return it->second;
    rt_material rec;
    std::memset(&rec, 0, sizeof rec);
    rec.texture = -1;
    m->describe(*this, rec);
    fs.materials.push_back(rec);
    int id = (int)fs.materials.size() - 1;
    mat_ids[m.get()] = id;
    return id;
}

// ---------------------------------------------------------------------------
// hittable.h / hittable_list.h / sphere.h / quad.h / triangle.h / bvh.h /
// constant_medium.h
// ---------------------------------------------------------------------------
class hittable {
  public:
    virtual ~hittable() = default;
    virtual aabb bounding_box() const = 0;
    virtual void flatten(rtb200::flattener& f) const = 0;
    // For bvh_node's replay of the reference's median split (SURVEY Q15), which only matters to
    // constant_medium objects: does this subtree hold one, and how many objects of the
    // reference's list does this object stand for (triangle_soup: one per triangle)?
    virtual bool has_medium() const { return false; }
    virtual size_t list_items() const { return 1; }
    virtual aabb list_item_box(size_t) const { return bounding_box(); }
};

class hittable_list : public hittable {
  public:
    std::vector<shared_ptr<hittable>> objects;
    hittable_list() {}
    hittable_list(shared_ptr<hittable> object) { add(object); }
    void clear() { objects.clear(); }
    void add(shared_ptr<hittable> object) {
        objects.push_back(object);
        bbox = aabb(bbox, object->bounding_box());
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override {
        for (const auto& o : objects) o->flatten(f);
    }
    bool has_medium() const override {
        for (const auto& o : objects)
            if (o->has_medium()) return true;
        return false;
    }
  private:
    aabb bbox;
};

class sphere : public hittable {
  public:
    sphere(const point3& static_center, double r, shared_ptr<material> m)
        : c0(static_center), cvec(0, 0, 0), radius(std::fmax(0, r)), mat(m) {
        vec3 rvec(r, r, r);
        bbox = aabb(static_center - rvec, static_center + rvec);
    }
    sphere(const point3& center1, const point3& center2, double r, shared_ptr<material> m)
        : c0(center1), cvec(center2 - center1), radius(std::fmax(0, r)), mat(m) {
        vec3 rvec(r, r, r);
        aabb b0(c0 - rvec, c0 + rvec);
        point3 c1 = c0 + 1.0 * cvec;
        aabb b1(c1 - rvec, c1 + rvec);
        bbox = aabb(b0, b1);
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override { f.add_sphere(c0, cvec, radius, mat); }
  private:
    point3 c0;
    vec3 cvec;
    double radius;
    shared_ptr<material> mat;
    aabb bbox;
};

class quad : public hittable {
  public:
    quad(const point3& q, const vec3& eu, const vec3& ev, shared_ptr<material> m) : Q(q), u(eu), v(ev), mat(m) {
        bbox = aabb(aabb(Q, Q + u + v), aabb(Q + u, Q + v));
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override { f.add_quad(Q, u, v, mat); }
  private:
    point3 Q;
    vec3 u, v;
    shared_ptr<material> mat;
    aabb bbox;
};

// quad.h:86-108 — same six sides in the same order
inline shared_ptr<hittable_list> box(const point3& a, const point3& b, shared_ptr<material> mat) {
    auto sides = make_shared<hittable_list>();
    point3 lo(std::fmin(a.x(), b.x()), std::fmin(a.y(), b.y()), std::fmin(a.z(), b.z()));
    point3 hi(std::fmax(a.x(), b.x()), std::fmax(a.y(), b.y()), std::fmax(a.z(), b.z()));
    vec3 dx(hi.x() - lo.x(), 0, 0), dy(0, hi.y() - lo.y(), 0), dz(0, 0, hi.z() - lo.z());
    sides->add(make_shared<quad>(point3(lo.x(), lo.y(), hi.z()), dx, dy, mat));   // front
    sides->add(make_shared<quad>(point3(hi.x(), lo.y(), hi.z()), -dz, dy, mat));  // right
    sides->add(make_shared<quad>(point3(hi.x(), lo.y(), lo.z()), -dx, dy, mat));  // back
    sides->add(make_shared<quad>(point3(lo.x(), lo.y(), lo.z()), dz, dy, mat));   // left
    sides->add(make_shared<quad>(point3(lo.x(), hi.y(), hi.z()), dx, -dz, mat));  // top
    sides->add(make_shared<quad>(point3(lo.x(), lo.y(), lo.z()), dx, dz, mat));   // bottom
    return sides;
}

class triangle : public hittable {
  public:
    triangle(vec3 a, vec3 b, vec3 c, std::shared_ptr<material> m) : p0(a), p1(b), p2(c), mat(m) {
        uv[0] = 0; uv[1] = 0; uv[2] = 1; uv[3] = 0; uv[4] = 0; uv[5] = 1;  // triangle.h:24-26
        set_bbox();
    }
    // triangle.h:30-44: the "wrap to [0,1)" at :40-42 assigns to the constructor
    // parameters, so the members keep the raw UVs (SURVEY Q4) — nothing to wrap here.
    triangle(vec3 a, vec3 b, vec3 c, std::shared_ptr<material> m, glm::vec2 t0, glm::vec2 t1, glm::vec2 t2)
        : p0(a), p1(b), p2(c), mat(m) {
        uv[0] = t0.x; uv[1] = t0.y; uv[2] = t1.x; uv[3] = t1.y; uv[4] = t2.x; uv[5] = t2.y;
        set_bbox();
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override { f.add_triangle(p0, p1, p2, uv, mat); }
  private:
    vec3 p0, p1, p2;
    std::shared_ptr<material> mat;
    float uv[6];
    aabb bbox;
    void set_bbox() {
        vec3 lo(std::min({p0.x(), p1.x(), p2.x()}), std::min({p0.y(), p1.y(), p2.y()}), std::min({p0.z(), p1.z(), p2.z()}));
        vec3 hi(std::max({p0.x(), p1.x(), p2.x()}), std::max({p0.y(), p1.y(), p2.y()}), std::max({p0.z(), p1.z(), p2.z()}));
        bbox = aabb(lo, hi);
    }
};

// triangle.h:146-169, including its `height + orig.x()` for the second vertex's y.
inline std::shared_ptr<hittable_list> triangle_quad(const point3& orig, double height, double width, shared_ptr<material> mat) {
    auto sides = make_shared<hittable_list>();
    sides->add(make_shared<triangle>(point3(orig), vec3(orig.x(), height + orig.x(), orig.z()),
                                     vec3(width + orig.x(), orig.y(), orig.z()), mat));
    sides->add(make_shared<triangle>(point3(orig.x() + width, orig.y(), orig.z()),
                                     vec3(orig.x() + width, orig.y() + height, orig.z()),
                                     vec3(orig.x(), height + orig.y(), orig.z()), mat));
    return sides;
}

// Many triangles of one material as ONE scene object (SURVEY 8f rank 2).  The reference's
// mesh.h:95-121 creates one shared_ptr<triangle> per face; a million-face OBJ then spends its load
// time in the allocator.  A soup stores the faces in the layout the C ABI wants and flattens with
// one append; it contributes its triangles to the canonical primitive numbering in order,
// exactly as that many separate `triangle` objects would.
class triangle_soup : public hittable {
  public:
    explicit triangle_soup(std::shared_ptr<material> m) : mat(m) {}
    void reserve(size_t n) { tris.reserve(n); }
    size_t size() const { return tris.size(); }
    // same arguments as the seven-argument triangle constructor (triangle.h:30-44)
    void add(const vec3& a, const vec3& b, const vec3& c, glm::vec2 t0, glm::vec2 t1, glm::vec2 t2) {
        rt_triangle t;
        std::memset(&t, 0, sizeof t);
        for (int k = 0; k < 3; k++) { t.p0[k] = a[k]; t.p1[k] = b[k]; t.p2[k] = c[k]; }
        t.uv0[0] = t0.x; t.uv0[1] = t0.y; t.uv1[0] = t1.x; t.uv1[1] = t1.y; t.uv2[0] = t2.x; t.uv2[1] = t2.y;
        t.material = -1;
        t.xform = -1;
        tris.push_back(t);
        for (int k = 0; k < 3; k++) {
            lo[k] = std::min({lo[k], a[k], b[k], c[k]});
            hi[k] = std::max({hi[k], a[k], b[k], c[k]});
        }
    }
    // bulk interface for loaders that fill the records from several threads
    static void fill(rt_triangle& t, const vec3& a, const vec3& b, const vec3& c, glm::vec2 t0, glm::vec2 t1, glm::vec2 t2) {
        std::memset(&t, 0, sizeof t);
        for (int k = 0; k < 3; k++) { t.p0[k] = a[k]; t.p1[k] = b[k]; t.p2[k] = c[k]; }
        t.uv0[0] = t0.x; t.uv0[1] = t0.y; t.uv1[0] = t1.x; t.uv1[1] = t1.y; t.uv2[0] = t2.x; t.uv2[1] = t2.y;
        t.material = -1;
        t.xform = -1;
    }
    rt_triangle* grow(size_t n) {
        tris.resize(tris.size() + n);
        return tris.data() + tris.size() - n;
    }
    void merge_bounds(const double l[3], const double h[3]) {
        for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], l[k]); hi[k] = std::max(hi[k], h[k]); }
    }
    aabb bounding_box() const override {
        if (tris.empty()) return aabb();
        return aabb(vec3(lo[0], lo[1], lo[2]), vec3(hi[0], hi[1], hi[2]));
    }
    void flatten(rtb200::flattener& f) const override { f.add_triangles(tris, mat); }
    size_t list_items() const override { return tris.size(); }
    aabb list_item_box(size_t k) const override {  // what triangle::set_bbox gives the k-th face
        const rt_triangle& t = tris[k];
        return aabb(vec3(std::min({t.p0[0], t.p1[0], t.p2[0]}), std::min({t.p0[1], t.p1[1], t.p2[1]}), std::min({t.p0[2], t.p1[2], t.p2[2]})),
                    vec3(std::max({t.p0[0], t.p1[0], t.p2[0]}), std::max({t.p0[1], t.p1[1], t.p2[1]}), std::max({t.p0[2], t.p1[2], t.p2[2]})));
    }
  private:
    std::shared_ptr<material> mat;
    rtb200::pod_vector<rt_triangle> tris;
    double lo[3] = {infinity, infinity, infinity}, hi[3] = {-infinity, -infinity, -infinity};
};

// The same faces as a triangle_soup, as an indexed mesh (rt_mesh): shared float vertices and 12 bytes of
// indices per triangle instead of 104 bytes of doubles.  Flattens to ONE rt_mesh and one world ref; the
// device records derived from it are bit-identical to the soup's, so is the image.
class indexed_mesh : public hittable {
  public:
    indexed_mesh(std::shared_ptr<const rtb200::mesh_arrays> arrays, std::shared_ptr<material> m, const double l[3], const double h[3])
        : data(std::move(arrays)), mat(std::move(m)) {
        for (int k = 0; k < 3; k++) { lo[k] = l[k]; hi[k] = h[k]; }
    }
    const rtb200::mesh_arrays& arrays() const { return *data; }
    aabb bounding_box() const override {
        if (data->triangles() == 0) return aabb();
        return aabb(vec3(lo[0], lo[1], lo[2]), vec3(hi[0], hi[1], hi[2]));
    }
    void flatten(rtb200::flattener& f) const override { f.add_mesh(data, mat); }
    size_t list_items() const override { return data->triangles(); }
    aabb list_item_box(size_t k) const override {  // what triangle::set_bbox gives the k-th face
        double p[3][3];
        for (int c = 0; c < 3; c++) data->corner(k, c, p[c]);
        return aabb(vec3(std::min({p[0][0], p[1][0], p[2][0]}), std::min({p[0][1], p[1][1], p[2][1]}), std::min({p[0][2], p[1][2], p[2][2]})),
                    vec3(std::max({p[0][0], p[1][0], p[2][0]}), std::max({p[0][1], p[1][1], p[2][1]}), std::max({p[0][2], p[1][2], p[2][2]})));
    }
  private:
    std::shared_ptr<const rtb200::mesh_arrays> data;
    std::shared_ptr<material> mat;
    double lo[3] = {infinity, infinity, infinity}, hi[3] = {-infinity, -infinity, -infinity};
};

class translate : public hittable {
  public:
    translate(shared_ptr<hittable> obj, const vec3& off) : object(obj), offset(off) { bbox = object->bounding_box() + offset; }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override {
        f.push_translate(offset);
        object->flatten(f);
        f.pop();
    }
    bool has_medium() const override { return object->has_medium(); }
  private:
    shared_ptr<hittable> object;
    vec3 offset;
    aabb bbox;
};

class rotate_y : public hittable {
  public:
    rotate_y(shared_ptr<hittable> obj, double angle) : object(obj) {
        double radians = degrees_to_radians(angle);
        sin_theta = std::sin(radians);
        cos_theta = std::cos(radians);
        aabb b = object->bounding_box();
        point3 lo(infinity, infinity, infinity), hi(-infinity, -infinity, -infinity);
        for (int i = 0; i < 2; i++)
            for (int j = 0; j < 2; j++)
                for (int k = 0; k < 2; k++) {
                    double x = i * b.x.max + (1 - i) * b.x.min;
                    double y = j * b.y.max + (1 - j) * b.y.min;
                    double z = k * b.z.max + (1 - k) * b.z.min;
                    vec3 corner(cos_theta * x + sin_theta * z, y, -sin_theta * x + cos_theta * z);
                    for (int c = 0; c < 3; c++) {
                        lo[c] = std::fmin(lo[c], corner[c]);
                        hi[c] = std::fmax(hi[c], corner[c]);
                    }
                }
        bbox = aabb(lo, hi);
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override {
        f.push_rotate_y(sin_theta, cos_theta);
        object->flatten(f);
        f.pop();
    }
    bool has_medium() const override { return object->has_medium(); }
  private:
    shared_ptr<hittable> object;
    double sin_theta, cos_theta;
    aabb bbox;
};

// The device builds its own SAH BVH, so a bvh_node contributes no structure.  What it
// must preserve is a side effect of the reference's build (bvh.h:24-44): an object that
// lands in a 1-object span becomes BOTH children (bvh.h:31-33) and is hit() twice per
// visit, which doubles the density of a constant_medium (SURVEY Q15).  The constructor
// replays the reference's longest-axis sort + median split on the same bounding boxes to
// find those objects and records a multiplicity per child.
class bvh_node : public hittable {
  public:
    // bvh.h:13-45.  The tree itself is rebuilt by rt_upload_scene; what survives of the
    // reference's median split is which list entries end up ALONE in a leaf, because such a leaf
    // stores its object as both children (bvh.h:31-33) and a constant_medium hit twice per visit
    // behaves like a medium of twice the density (SURVEY Q15).  The split is replayed only when the
    // list holds a medium at all; an object that stands for many list entries (triangle_soup)
    // takes part with one box per entry, exactly as that many `triangle` objects would.
    bvh_node(hittable_list list) {
        originals = list.objects;
        mult.assign(originals.size(), 1);
        bbox = aabb::empty();
        bool sensitive = false;
        for (const auto& o : originals) {
            bbox = aabb(bbox, o->bounding_box());
            sensitive = sensitive || o->has_medium();
        }
        if (!sensitive || originals.empty()) return;
        size_t n = 0;
        for (const auto& o : originals) n += o->list_items();
        items.reserve(n);
        for (size_t i = 0; i < originals.size(); i++) {
            const size_t k = originals[i]->list_items();
            if (k == 1) items.push_back({originals[i]->list_item_box(0), (int)i});
            else for (size_t j = 0; j < k; j++) items.push_back({originals[i]->list_item_box(j), -1});
        }
        if (!items.empty()) replay(0, items.size());
        std::vector<item>().swap(items);
    }
    aabb bounding_box() const override { return bbox; }
    void flatten(rtb200::flattener& f) const override {
        for (size_t i = 0; i < originals.size(); i++) {
            int saved = f.multiplicity;
            f.multiplicity = saved * mult[i];
            originals[i]->flatten(f);
            f.multiplicity = saved;
        }
    }
    bool has_medium() const override {
        for (const auto& o : originals)
            if (o->has_medium()) return true;
        return false;
    }
    int multiplicity_of(size_t insertion_index) const { return mult[insertion_index]; }
  private:
    struct item { aabb box; int index; };  // index < 0: one of many entries of a bulk object
    std::vector<item> items;
    std::vector<shared_ptr<hittable>> originals;
    std::vector<int> mult;
    aabb bbox;

    void replay(size_t start, size_t end) {
        aabb span_box = aabb::empty();
        for (size_t i = start; i < end; i++) span_box = aabb(span_box, items[i].box);
        const int axis = span_box.longest_axis();
        const size_t span = end - start;
        if (span == 1) {
            if (items[start].index >= 0) mult[items[start].index] *= 2;
            return;
        }
        if (span == 2) return;
        std::sort(items.begin() + start, items.begin() + end, [axis](const item& a, const item& b) {
            return a.box.axis_interval(axis).min < b.box.axis_interval(axis).min;
        });
        const size_t mid = start + span / 2;
        replay(start, mid);
        replay(mid, end);
    }
};

class constant_medium : public hittable {
  public:
    constant_medium(shared_ptr<hittable> b, double d, shared_ptr<texture> tex)
        : boundary(b), density(d), phase_function(make_shared<isotropic>(tex)) {}
    constant_medium(shared_ptr<hittable> b, double d, const color& albedo)
        : boundary(b), density(d), phase_function(make_shared<isotropic>(albedo)) {}
    aabb bounding_box() const override { return boundary->bounding_box(); }
    void flatten(rtb200::flattener& f) const override { f.add_medium(*boundary, density, phase_function); }
    bool has_medium() const override { return true; }
  private:
    shared_ptr<hittable> boundary;
    double density;
    shared_ptr<material> phase_function;
};

inline void rtb200::flattener::add_medium(const hittable& boundary, double density, const shared_ptr<material>& phase) {
    rt_medium m;
    std::memset(&m, 0, sizeof m);
    m.boundary_first = (int)fs.boundary_refs.size();
    int saved_mult = multiplicity;
    boundary_depth++;
    boundary.flatten(*this);  // a medium nested in a boundary is ignored by add_ref's routing
    boundary_depth--;
    multiplicity = saved_mult;
    m.boundary_count = (int)fs.boundary_refs.size() - m.boundary_first;
    m.density = density;
    m.multiplicity = multiplicity;
    m.material = material_id(phase);
    m.xform = current_xform();
    if (boundary_depth == 0) fs.media.push_back(m);
}

// ---------------------------------------------------------------------------
// mesh.h — OBJ loader that pushes triangles straight into the world list
// ---------------------------------------------------------------------------
class mesh {
  public:
    mesh() {}
    mesh(const std::vector<glm::mat4>& tris) : mesh_matrices(tris) {}

    // mesh.h:22-92.  Understands `v`, `vt` and `f a/b/c ...` records; 3- and 4-vertex
    // faces.  A 4-vertex face becomes (0,1,2) and (0,2,3) but BOTH halves take the UVs
    // of the face's first three corners (mesh.h:78-81 passes the same uv index list and
    // addTriangle reads entries [0],[1],[2]; SURVEY Q5).  Vertex positions go through
    // the float mat4 before being widened to double (mesh.h:105-117).
    // Which loader loadObj uses.  false (default): the fast path -- the file is read in one piece,
    // numbers are parsed with std::from_chars (correctly rounded, like operator>>), and the faces go
    // into ONE triangle_soup object.  true: the reference's own structure (mesh.h:22-92) -- a
    // stringstream per line and one shared_ptr<triangle> per face.  Both give the same flattened
    // scene, byte for byte (tests/test_obj_fast_path.py).
    static bool& per_triangle_objects() {
        static bool flag = false;
        return flag;
    }
    // With the fast path: true makes the faces ONE indexed_mesh (rt_mesh: each vertex transformed once, stored
    // as float, 12 bytes of indices per triangle) instead of a triangle_soup -- same faces, same order, same
    // skip rules and UVs (Q5), same device records and image.  Default false.
    static bool& indexed_meshes() {
        static bool flag = false;
        return flag;
    }

    bool loadObj(const std::string path, hittable_list& world, const shared_ptr<lambertian> mat, glm::mat4 transform) {
        return per_triangle_objects() ? loadObjReference(path, world, mat, transform) : loadObjFast(path, world, mat, transform);
    }

    // mesh.h:22-92.  Understands `v`, `vt` and `f a/b/c ...` records; 3- and 4-vertex
    // faces.  A 4-vertex face becomes (0,1,2) and (0,2,3) but BOTH halves take the UVs
    // of the face's first three corners (mesh.h:78-81 passes the same uv index list and
    // addTriangle reads entries [0],[1],[2]; SURVEY Q5).  Vertex positions go through
    // the float mat4 before being widened to double (mesh.h:105-117).
    bool loadObjReference(const std::string path, hittable_list& world, const shared_ptr<lambertian> mat, glm::mat4 transform) {
        std::ifstream file(path);
        if (!file.is_open()) {
            std::cerr << "Failed to open file: " << path << std::endl;
            return false;
        }
        std::vector<glm::vec3> positions;
        std::vector<glm::vec2> texcoords;
        std::string line;
        while (std::getline(file, line)) {
            std::istringstream ss(line);
            std::string tag;
            ss >> tag;
            if (tag == "v") {
                glm::vec3 p;
                ss >> p.x >> p.y >> p.z;
                positions.push_back(p);
            } else if (tag == "vt") {
                glm::vec2 t;
                ss >> t.x >> t.y;
                texcoords.push_back(t);
            } else if (tag == "f") {
                std::vector<int> vi, ti;
                std::string corner;
                while (ss >> corner) {
                    std::istringstream cs(corner);
                    int v = 0, vt = 0, vn = 0;
                    char slash;
                    cs >> v >> slash >> vt >> slash >> vn;
                    vi.push_back(v - 1);
                    ti.push_back(vt - 1);
                }
                if (vi.size() < 3) continue;
                if (vi.size() == 3) {
                    addTriangle(positions, texcoords, vi[0], vi[1], vi[2], ti, mat, world, transform);
                } else if (vi.size() == 4) {
                    addTriangle(positions, texcoords, vi[0], vi[1], vi[2], ti, mat, world, transform);
                    addTriangle(positions, texcoords, vi[0], vi[2], vi[3], ti, mat, world, transform);
                } else {
                    std::cerr << "Skipping face with " << vi.size() << " vertices." << std::endl;
                }
            }
        }
        return true;
    }

    // The same records from the same file, without the per-line streams and per-face objects:
    // the file is cut at line ends into one piece per host thread; every piece is parsed into its
    // own vertex / texcoord / face lists (OBJ indices are absolute, so the pieces are independent),
    // the lists are joined in file order, and the triangles are then written in parallel.
    struct obj_piece {
        std::vector<glm::vec3> positions;
        std::vector<glm::vec2> texcoords;
        std::vector<int> face;  // per face: count (3 or 4), v0..v3, t0..t2
        size_t triangles = 0, first_triangle = 0;
        double lo[3] = {infinity, infinity, infinity}, hi[3] = {-infinity, -infinity, -infinity};
    };

    static void parse_obj_piece(const char* p, const char* end, obj_piece& out) {
        auto is_space = [](char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; };
        // operator>>(float): skips blanks, parses the longest valid number, leaves 0 on failure
        auto read_float = [&](const char*& q, const char* e, float& v) {
            while (q < e && is_space(*q)) q++;
            const char* s = q;
            if (s < e && *s == '+') s++;  // from_chars does not accept a leading '+', streams do
            float x = 0.0f;
            auto r = std::from_chars(s, e, x);
            if (r.ec != std::errc() && r.ec != std::errc::result_out_of_range) return false;
            v = x;
            q = r.ptr;
            return true;
        };
        auto read_int = [&](const char*& q, const char* e, int& v) {
            const char* s = q;
            if (s < e && *s == '+') s++;
            int x = 0;
            auto r = std::from_chars(s, e, x);
            if (r.ec != std::errc()) return false;
            v = x;
            q = r.ptr;
            return true;
        };
        out.positions.reserve((size_t)(end - p) / 64);
        out.texcoords.reserve((size_t)(end - p) / 64);
        out.face.reserve((size_t)(end - p) / 8);
        int vi[5], ti[5];
        while (p < end) {
            const char* eol = (const char*)std::memchr(p, '\n', (size_t)(end - p));
            const char* e = eol ? eol : end;
            const char* q = p;
            while (q < e && is_space(*q)) q++;
            const char* tag = q;
            while (q < e && !is_space(*q)) q++;
            const size_t tl = (size_t)(q - tag);
            if (tl == 1 && tag[0] == 'v') {
                glm::vec3 v;
                if (read_float(q, e, v.x) && read_float(q, e, v.y)) read_float(q, e, v.z);
                out.positions.push_back(v);
            } else if (tl == 2 && tag[0] == 'v' && tag[1] == 't') {
                glm::vec2 t;
                if (read_float(q, e, t.x)) read_float(q, e, t.y);
                out.texcoords.push_back(t);
            } else if (tl == 1 && tag[0] == 'f') {
                int n = 0;
                while (true) {
                    while (q < e && is_space(*q)) q++;
                    if (q >= e) break;
                    const char* ce = q;
                    while (ce < e && !is_space(*ce)) ce++;
                    // cs >> v >> slash >> vt >> slash >> vn: every step only runs if the one before worked
                    int v = 0, vt = 0;
                    const char* c = q;
                    if (read_int(c, ce, v) && c < ce) {
                        c++;  // the separator (any character, as `char slash` accepts)
                        read_int(c, ce, vt);
                    }
                    if (n < 5) { vi[n] = v - 1; ti[n] = vt - 1; }
                    n++;
                    q = ce;
                }
                if (n == 3 || n == 4) {
                    const int rec[8] = {n, vi[0], vi[1], vi[2], n == 4 ? vi[3] : -1, ti[0], ti[1], ti[2]};
                    out.face.insert(out.face.end(), rec, rec + 8);
                } else if (n > 4) {
                    std::cerr << "Skipping face with " << n << " vertices." << std::endl;
                }
            }
            p = eol ? eol + 1 : end;
        }
    }

    bool loadObjFast(const std::string& path, hittable_list& world, const shared_ptr<lambertian>& mat, const glm::mat4& transform) {
        rtb200::mapped_file file(path.c_str());
        if (!file.ok()) {
            std::cerr << "Failed to open file: " << path << std::endl;
            return false;
        }
        const char* const text = file.data();
        const size_t got = file.size();

        // ---- phase 1: parse, one piece per thread ------------------------------------------------
        const size_t n_pieces = rtb200::host_parts(got, 1u << 20);
        std::vector<size_t> cut(n_pieces + 1, got);
        cut[0] = 0;
        for (size_t i = 1; i < n_pieces; i++) {
            size_t at = std::max(cut[i - 1], got * i / n_pieces);
            const void* nl = at < got ? std::memchr(text + at, '\n', got - at) : nullptr;
            cut[i] = nl ? (size_t)((const char*)nl - text) + 1 : got;
        }
        std::vector<obj_piece> pieces(n_pieces);
        auto for_pieces = [&](auto&& fn) { rtb200::parallel_parts(n_pieces, [&fn](size_t i, size_t) { fn(i); }); };
        for_pieces([&](size_t i) { parse_obj_piece(text + cut[i], text + cut[i + 1], pieces[i]); });

        // ---- join the vertex lists in file order -----------------------------------------------------
        std::vector<glm::vec3> positions;
        std::vector<glm::vec2> texcoords;
        {
            size_t np = 0, nt = 0;
            for (const obj_piece& pc : pieces) { np += pc.positions.size(); nt += pc.texcoords.size(); }
            positions.reserve(np);
            texcoords.reserve(nt);
            for (obj_piece& pc : pieces) {
                positions.insert(positions.end(), pc.positions.begin(), pc.positions.end());
                texcoords.insert(texcoords.end(), pc.texcoords.begin(), pc.texcoords.end());
                std::vector<glm::vec3>().swap(pc.positions);
                std::vector<glm::vec2>().swap(pc.texcoords);
            }
        }
        // ---- phase 2: count the triangles of every piece, then write them in parallel -------------------
        const int nv = (int)positions.size();
        auto face_ok = [&](const int* r, int a, int b, int c) {
            const int v0 = r[1 + a], v1 = r[1 + b], v2 = r[1 + c];
            return v0 >= 0 && v1 >= 0 && v2 >= 0 && v0 < nv && v1 < nv && v2 < nv;
        };
        for_pieces([&](size_t i) {
            obj_piece& pc = pieces[i];
            for (size_t k = 0; k + 8 <= pc.face.size(); k += 8) {
                const int* r = &pc.face[k];
                pc.triangles += face_ok(r, 0, 1, 2) ? 1 : 0;
                if (r[0] == 4) pc.triangles += face_ok(r, 0, 2, 3) ? 1 : 0;
            }
        });
        size_t total = 0, listed = 0;
        for (obj_piece& pc : pieces) {
            pc.first_triangle = total;
            total += pc.triangles;
            for (size_t k = 0; k + 8 <= pc.face.size(); k += 8) listed += pc.face[k] == 4 ? 2 : 1;
        }
        // the reference indexes vertices[] unchecked (undefined behaviour); such faces are refused here
        if (listed != total) std::cerr << "Skipping " << (listed - total) << " triangles with a vertex index outside the file." << std::endl;
        if (total == 0) return true;
        if (indexed_meshes()) return emitIndexed(pieces, positions, texcoords, total, world, mat, transform);
        auto soup = make_shared<triangle_soup>(mat);
        rt_triangle* out = soup->grow(total);
        const size_t m0 = mesh_matrices.size();
        mesh_matrices.resize(m0 + total);
        for_pieces([&](size_t i) {
            obj_piece& pc = pieces[i];
            size_t w = pc.first_triangle;
            auto emit = [&](const int* r, int a, int b, int c) {
                if (!face_ok(r, a, b, c)) return;
                // mesh.h:105-117: float mat4 times float position, widened to double afterwards
                glm::vec4 A = transform * glm::vec4(positions[r[1 + a]], 1.0f);
                glm::vec4 B = transform * glm::vec4(positions[r[1 + b]], 1.0f);
                glm::vec4 C = transform * glm::vec4(positions[r[1 + c]], 1.0f);
                glm::mat4 m(1.0f);
                m[0] = A; m[1] = B; m[2] = C; m[3] = glm::vec4(0, 0, 0, 1);
                mesh_matrices[m0 + w] = m;
                auto uv_at = [&](int k) {  // always the face's FIRST three texcoord indices (SURVEY Q5)
                    int idx = r[5 + k];
                    return (idx >= 0 && idx < (int)texcoords.size()) ? texcoords[idx] : glm::vec2(0, 0);
                };
                const vec3 a3(A.x, A.y, A.z), b3(B.x, B.y, B.z), c3(C.x, C.y, C.z);
                triangle_soup::fill(out[w], a3, b3, c3, uv_at(0), uv_at(1), uv_at(2));
                for (int k = 0; k < 3; k++) {
                    pc.lo[k] = std::min({pc.lo[k], a3[k], b3[k], c3[k]});
                    pc.hi[k] = std::max({pc.hi[k], a3[k], b3[k], c3[k]});
                }
                w++;
            };
            for (size_t k = 0; k + 8 <= pc.face.size(); k += 8) {
                const int* r = &pc.face[k];
                emit(r, 0, 1, 2);
                if (r[0] == 4) emit(r, 0, 2, 3);
            }
        });
        for (const obj_piece& pc : pieces) soup->merge_bounds(pc.lo, pc.hi);
        world.add(soup);
        return true;
    }

    // loadObjFast's faces as one indexed_mesh.  Every vertex goes through the float mat4 once (the soup
    // transforms it once per face that uses it: the same operation, the same floats).  Texture coordinates
    // keep their own indices; a corner whose `vt` index is missing or out of range points at a (0,0)
    // appended after the file's own, which is the UV the soup gives it.
    bool emitIndexed(std::vector<obj_piece>& pieces, const std::vector<glm::vec3>& positions, const std::vector<glm::vec2>& texcoords,
                     size_t total, hittable_list& world, const shared_ptr<lambertian>& mat, const glm::mat4& transform) {
        auto for_pieces = [&](auto&& fn) { rtb200::parallel_parts(pieces.size(), [&fn](size_t i, size_t) { fn(i); }); };
        const size_t nv = positions.size(), nt = texcoords.size();
        auto a = std::make_shared<rtb200::mesh_arrays>();
        std::vector<glm::vec4> moved(nv);
        a->positions.resize(3 * nv);
        rtb200::parallel_parts(rtb200::host_parts(nv, 1 << 16), [&](size_t part, size_t parts) {
            for (size_t v = nv * part / parts, e = nv * (part + 1) / parts; v < e; v++) {
                moved[v] = transform * glm::vec4(positions[v], 1.0f);  // mesh.h:105-117
                a->positions[3 * v] = moved[v].x; a->positions[3 * v + 1] = moved[v].y; a->positions[3 * v + 2] = moved[v].z;
            }
        });
        a->uvs.resize(2 * (nt + 1));
        for (size_t t = 0; t < nt; t++) { a->uvs[2 * t] = texcoords[t].x; a->uvs[2 * t + 1] = texcoords[t].y; }
        a->uvs[2 * nt] = 0.0f;
        a->uvs[2 * nt + 1] = 0.0f;
        a->indices.resize(3 * total);
        a->uv_indices.resize(3 * total);
        const size_t m0 = mesh_matrices.size();
        mesh_matrices.resize(m0 + total);
        const int nvi = (int)nv;
        for_pieces([&](size_t i) {
            obj_piece& pc = pieces[i];
            size_t w = pc.first_triangle;
            auto emit = [&](const int* r, int a0, int b0, int c0) {
                const int v[3] = {r[1 + a0], r[1 + b0], r[1 + c0]};
                for (int k = 0; k < 3; k++)
                    if (v[k] < 0 || v[k] >= nvi) return;
                glm::mat4 m(1.0f);
                for (int k = 0; k < 3; k++) {
                    a->indices[3 * w + k] = (uint32_t)v[k];
                    const int t = r[5 + k];  // always the face's FIRST three texcoord indices (SURVEY Q5)
                    a->uv_indices[3 * w + k] = (t >= 0 && t < (int)nt) ? (uint32_t)t : (uint32_t)nt;
                    m[k] = moved[(size_t)v[k]];
                    const double p[3] = {moved[(size_t)v[k]].x, moved[(size_t)v[k]].y, moved[(size_t)v[k]].z};
                    for (int d = 0; d < 3; d++) { pc.lo[d] = std::min(pc.lo[d], p[d]); pc.hi[d] = std::max(pc.hi[d], p[d]); }
                }
                m[3] = glm::vec4(0, 0, 0, 1);
                mesh_matrices[m0 + w] = m;
                w++;
            };
            for (size_t k = 0; k + 8 <= pc.face.size(); k += 8) {
                const int* r = &pc.face[k];
                emit(r, 0, 1, 2);
                if (r[0] == 4) emit(r, 0, 2, 3);
            }
        });
        double lo[3] = {infinity, infinity, infinity}, hi[3] = {-infinity, -infinity, -infinity};
        for (const obj_piece& pc : pieces)
            for (int k = 0; k < 3; k++) { lo[k] = std::min(lo[k], pc.lo[k]); hi[k] = std::max(hi[k], pc.hi[k]); }
        world.add(make_shared<indexed_mesh>(std::move(a), mat, lo, hi));
        return true;
    }

    void addTriangle(const std::vector<glm::vec3>& vertices, const std::vector<glm::vec2>& uvs, int v0, int v1, int v2,
                     const std::vector<int>& uv_indices, const shared_ptr<lambertian> mat, hittable_list& world,
                     const glm::mat4& transform) {
        glm::vec4 a = transform * glm::vec4(vertices[v0], 1.0f);
        glm::vec4 b = transform * glm::vec4(vertices[v1], 1.0f);
        glm::vec4 c = transform * glm::vec4(vertices[v2], 1.0f);
        glm::mat4 m(1.0f);
        m[0] = a; m[1] = b; m[2] = c; m[3] = glm::vec4(0, 0, 0, 1);
        mesh_matrices.push_back(m);
        // the reference indexes uvs[] unchecked; a face without texture coordinates
        // would read out of bounds there — here it gets (0,0)
        auto uv_at = [&](int k) {
            int idx = uv_indices[k];
            return (idx >= 0 && idx < (int)uvs.size()) ? uvs[idx] : glm::vec2(0, 0);
        };
        world.add(make_shared<triangle>(vec3(a.x, a.y, a.z), vec3(b.x, b.y, b.z), vec3(c.x, c.y, c.z), mat, uv_at(0),
                                        uv_at(1), uv_at(2)));
    }

    void applyTransform(const glm::mat4& t) {
        for (auto& m : mesh_matrices)
            for (int i = 0; i < 3; ++i) m[i] = t * m[i];
    }
    void scale(float factor) { applyTransform(glm::scale(glm::mat4(1.0f), glm::vec3(factor))); }
    void rotate(float angle, const glm::vec3& axis) { applyTransform(glm::rotate(glm::mat4(1.0f), glm::radians(angle), axis)); }
    void translate(const glm::vec3& offset) { applyTransform(glm::translate(glm::mat4(1.0f), offset)); }

    std::vector<glm::mat4> mesh_matrices;
};

// ---------------------------------------------------------------------------
// point_light.h
// ---------------------------------------------------------------------------
class point_light {
  public:
    point_light(point3 p, color i, double s) : position(p), intensity(i), size(s) {}
    point3 get_position() const { return position; }
    color get_intensity() const { return intensity; }
    double get_size() const { return size; }
  private:
    point3 position;
    color intensity;
    double size;
};

// ---------------------------------------------------------------------------
// camera.h (Camera.txt) — same public fields; render() drives the CUDA library
// ---------------------------------------------------------------------------
namespace rtb200 {

inline void flatten_scene(const hittable& world, const std::vector<point_light>& lights, flat_scene& fs) {
    flattener f(fs);
    world.flatten(f);
    for (size_t i = 0; i < fs.images.size(); i++) fs.images[i].rgb = fs.image_bytes[i].data();
    for (const auto& l : lights) {
        rt_point_light pl;
        for (int k = 0; k < 3; k++) { pl.position[k] = l.get_position()[k]; pl.intensity[k] = l.get_intensity()[k]; }
        pl.size = l.get_size();
        fs.lights.push_back(pl);
    }
}

bool write_png_rgb8(const char* path, int w, int h, const uint8_t* rgb);  // png_write.h

}  // namespace rtb200

class camera {
  public:
    // Camera.txt:39-40 declares these two `const` (1024, 16:9); they are plain
    // members here so that other frame sizes are expressible (SURVEY F5).
    int image_width = 1024;
    double aspect_ratio = 16.0 / 9.0;
    const char* image_name = "Default Image";
    int samples_per_pixel = 10;
    int max_depth = 10;
    color background = vec3(0, 0, 0);

    double vfov = 90;
    point3 lookfrom = point3(0, 0, 0);
    point3 lookat = point3(0, 0, -1);
    vec3 vup = vec3(0, 1, 0);

    double defocus_angle = 0;
    double focus_dist = 10;

    // additions (not in the reference): device(s), seed, and whether to write the PNG.  `devices` non-empty: the frame is
    // split over these GPUs of the box by ONE context (tile t -> devices[t mod n], tiles gathered over NVLink: replaces
    // the row bands over CPU threads of Camera.txt:59-61, 96-100); the image does not depend on how many there are
    int device = 0;
    std::vector<int> devices;
    uint64_t seed = 1;
    bool write_image = true;
    rt_stats last_stats{};
    std::vector<uint8_t> last_rgb8;
    // additions for SURVEY 8f rank 3 (download side): linear-radiance output and resumable renders.
    //   linear_name      "x.exr" / "x.pfm": also write the averaged linear radiance (before gamma)
    //   checkpoint_path  if the file exists and matches (scene, frame, depth, seed) the render
    //                    CONTINUES from the samples it holds; it is rewritten every
    //                    checkpoint_every_spp samples (0: only when the render stops early)
    //   stop_after_spp   > 0: stop once this many samples are in the frame (an orderly
    //                    interruption: checkpoint written, image of the samples so far)
    //   next_event_estimation  opt-in (SURVEY 8f rank 4): sample the quad emitters directly at diffuse
    //                    and isotropic vertices (RT_FLAG_NEE); same converged image, far less noise
    bool next_event_estimation = false;
    //   shadowed_point_lights  opt-in: shadow rays for the point lights (RT_FLAG_SHADOWED_POINT_LIGHTS);
    //                    the reference's are unshadowed (Camera.txt:240-272), so this changes the image
    bool shadowed_point_lights = false;
    std::string linear_name;
    std::string checkpoint_path;
    int checkpoint_every_spp = 0;
    int stop_after_spp = 0;
    int last_spp_done = 0;     // samples per pixel in the frame when render() returned
    int last_spp_resumed = 0;  // of which came from the checkpoint
    std::vector<float> last_linear;
    // per-pixel noise (RT_FLAG_MOMENTS; on only when one of the first two is set -- otherwise flags, passes and
    // checkpoint files are as without them):
    //   noise_target     > 0: stop once rms_std_error / mean_radiance of rt_frame_noise <= this, samples_per_pixel
    //                    being the cap
    //   noise_check_every_spp  the noise is checked only when the frame holds a multiple of this many samples, so the
    //                    stopping sample count is a function of the scene and settings alone, on any device list
    //   variance_name    "x.exr" / "x.pfm": also write the per-pixel sample variance (rt_download_variance)
    //   last_noise       rms_std_error / mean_radiance when render() returned (0 without moments)
    double noise_target = 0;
    int noise_check_every_spp = 256;
    std::string variance_name;
    double last_noise = 0;
    // turntable (rt_render_views): turntable_frames > 1 renders that many views of the scene in one batch, frame k from
    // lookfrom rotated about the axis through lookat along vup by 2 pi k / turntable_frames (turntable_camera), every
    // frame with `seed`; frame k is written to <stem>_<k:03d><ext> and last_rgb8 holds all frames, frame-major.  Not
    // combined with a checkpoint, a noise target, variance output or several devices.  0 or 1: off.
    int turntable_frames = 0;

    int image_height() const {
        int h = int(image_width / aspect_ratio);  // Camera.txt:137-138
        return h < 1 ? 1 : h;
    }

    void export_camera(rt_camera& c) const {
        for (int k = 0; k < 3; k++) {
            c.lookfrom[k] = lookfrom[k]; c.lookat[k] = lookat[k]; c.vup[k] = vup[k]; c.background[k] = background[k];
        }
        c.vfov = vfov; c.defocus_angle = defocus_angle; c.focus_dist = focus_dist;
    }

    // The rt_camera of turntable frame k (of turntable_frames), in double; frame 0 is the camera itself.
    rt_camera turntable_camera(int k) const {
        rt_camera c;
        export_camera(c);
        const int n = std::max(1, turntable_frames);
        if (k % n == 0) return c;
        const double pi = 3.1415926535897932385, angle = 2.0 * pi * (double)k / (double)n;
        double a[3] = {vup[0], vup[1], vup[2]};
        const double len = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
        for (double& x : a) x /= len;
        const double r[3] = {c.lookfrom[0] - c.lookat[0], c.lookfrom[1] - c.lookat[1], c.lookfrom[2] - c.lookat[2]};
        // Rodrigues: r cos + (a x r) sin + a (a . r)(1 - cos)
        const double cs = std::cos(angle), sn = std::sin(angle), ad = a[0] * r[0] + a[1] * r[1] + a[2] * r[2];
        const double ax[3] = {a[1] * r[2] - a[2] * r[1], a[2] * r[0] - a[0] * r[2], a[0] * r[1] - a[1] * r[0]};
        for (int i = 0; i < 3; i++) c.lookfrom[i] = c.lookat[i] + (r[i] * cs + ax[i] * sn + a[i] * ad * (1.0 - cs));
        return c;
    }

    // <stem>_<k:03d><ext> of a turntable frame (the extension is what follows the last '.' of the file name)
    static std::string frame_name(const std::string& name, int k) {
        const size_t slash = name.find_last_of("/\\"), dot = name.find_last_of('.');
        const bool ext = dot != std::string::npos && (slash == std::string::npos || dot > slash);
        char num[16];
        std::snprintf(num, sizeof num, "_%03d", k);
        return ext ? name.substr(0, dot) + num + name.substr(dot) : name + num;
    }

    // Same signature as Camera.txt:54.  Fails loudly (message + exit code 2) when the
    // CUDA path is unavailable — there is no CPU fallback.
    void render(const hittable& world, std::vector<point_light>& lights) {
        rtb200::flat_scene fs;
        rtb200::flatten_scene(world, lights, fs);
        export_camera(fs.camera);
        rt_scene_desc d = fs.desc();

        rt_ctx* ctx = nullptr;
        std::vector<int> devs = devices.empty() ? std::vector<int>{device} : devices;
        auto fail = [&](const char* what) {
            std::cerr << "\nrt_b200: " << what << " failed: " << (ctx ? rt_last_error(ctx) : "no context") << std::endl;
            if (ctx) rt_destroy(ctx);
            std::exit(2);
        };
        if (turntable_frames > 1 && (!checkpoint_path.empty() || noise_target > 0 || !variance_name.empty() || devs.size() > 1)) {
            std::cerr << "rt_b200: a turntable renders on one device without a checkpoint, a noise target or variance output" << std::endl;
            std::exit(2);
        }
        if (rt_create(&ctx, devs.data(), (int)devs.size()) != RT_OK) fail("rt_create");
        if (rt_upload_scene(ctx, &d) != RT_OK) fail("rt_upload_scene");
        if (turntable_frames > 1) {
            render_turntable(ctx, fail);
            return;
        }

        rt_render_params p;
        std::memset(&p, 0, sizeof p);
        p.struct_size = sizeof p;
        p.width = image_width;
        p.height = image_height();
        p.max_depth = max_depth;
        p.seed = seed;
        // resume: the frame so far is the checkpoint's integer sums
        int done = 0;
        rtb200::checkpoint_header ck;
        std::memset(&ck, 0, sizeof ck);
        std::memcpy(ck.magic, "RTB2CKPT", 8);
        const bool moments = noise_target > 0 || !variance_name.empty();
        ck.version = moments ? 2 : 1;  // 2: the second moments follow the sums
        ck.width = p.width; ck.height = p.height; ck.max_depth = max_depth; ck.seed = seed;
        ck.scene_hash = checkpoint_path.empty() ? 0 : fs.hash();
        const uint32_t estimator_flags = (next_event_estimation ? RT_FLAG_NEE : 0u) | (shadowed_point_lights ? RT_FLAG_SHADOWED_POINT_LIGHTS : 0u);
        ck.flags = estimator_flags;
        // a sample is clamped to 2^20 and stored in 2^-28 units: 2^16 samples of a saturated channel fill the 64-bit sum
        if (samples_per_pixel > 65536) {
            std::cerr << "rt_b200: samples_per_pixel " << samples_per_pixel << " exceeds 65536, the capacity of the 64-bit fixed-point sums" << std::endl;
            if (ctx) rt_destroy(ctx);
            std::exit(2);
        }
        if (moments && devs.size() > 1) {
            if (!checkpoint_path.empty()) {
                std::cerr << "rt_b200: a noise target or variance output with a checkpoint needs one device (moments are downloaded from one context device)" << std::endl;
                rt_destroy(ctx);
                std::exit(2);
            }
            p.shard_mode = RT_SHARD_TILES;  // a multi-device context resolves the noise of tile-sharded frames
        }
        std::vector<uint64_t> sums, msums;
        if (!checkpoint_path.empty()) {
            rtb200::checkpoint_header old;
            if (rtb200::read_checkpoint(checkpoint_path.c_str(), old, sums, &msums)) {
                if (moments && old.version != 2) {
                    std::cerr << "Ignoring " << checkpoint_path << ": it holds no second moments (version 1), which a noise target or variance output needs" << std::endl;
                } else if (old.width == ck.width && old.height == ck.height && old.max_depth == ck.max_depth && old.seed == ck.seed &&
                    old.scene_hash == ck.scene_hash && old.flags == ck.flags && old.spp_done <= samples_per_pixel) {
                    if (rt_accum_upload(ctx, sums.data(), sums.size() * 8, p.width, p.height) != RT_OK) fail("rt_accum_upload");
                    if (moments && rt_moments_upload(ctx, msums.data(), msums.size() * 8, p.width, p.height) != RT_OK) fail("rt_moments_upload");
                    done = old.spp_done;
                    std::cerr << "Resuming " << image_name << " at sample " << done << " from " << checkpoint_path << std::endl;
                } else {
                    std::cerr << "Ignoring " << checkpoint_path << ": it belongs to a different scene, frame, depth, seed or estimator (NEE / shadowed lights)" << std::endl;
                }
            }
        }
        last_spp_resumed = done;
        auto save_checkpoint = [&](int spp_done) {
            sums.resize((size_t)p.width * p.height * 4);
            if (rt_accum_download(ctx, sums.data(), sums.size() * 8) != RT_OK) fail("rt_accum_download");
            if (moments) {
                msums.resize((size_t)p.width * p.height * 6);
                if (rt_moments_download(ctx, msums.data(), msums.size() * 8) != RT_OK) fail("rt_moments_download");
            }
            ck.spp_done = spp_done;
            if (!rtb200::write_checkpoint(checkpoint_path.c_str(), ck, sums.data(), msums.data()))
                std::cerr << "\nrt_b200: cannot write checkpoint " << checkpoint_path << std::endl;
        };
        // progressive passes so the reference's progress line (Camera.txt:102-106) still ticks
        const int target = stop_after_spp > 0 ? std::min(stop_after_spp, samples_per_pixel) : samples_per_pixel;
        const int pass_spp = std::max(1, std::min(samples_per_pixel, 64));
        int since_save = 0, passes = 0;
        bool fresh = done == 0, converged = false;
        const int check_every = std::max(1, noise_check_every_spp);
        auto frame_noise = [&]() {
            double mean = 0, rms = 0;
            if (rt_frame_noise(ctx, done, &mean, &rms) != RT_OK) fail("rt_frame_noise");
            return mean > 0 ? rms / mean : 0.0;
        };
        while (done < target && !converged) {
            int n = std::min(pass_spp, target - done);
            if (!checkpoint_path.empty() && checkpoint_every_spp > 0) n = std::min(n, std::max(1, checkpoint_every_spp - since_save));
            if (noise_target > 0) n = std::min(n, check_every - done % check_every);
            p.samples_per_pixel = n;
            p.spp_begin = done;
            // passes after the first are enqueued without waiting and overlap their drains (RT_FLAG_OVERLAP: the last,
            // longest paths of one pass run while the next fills the freed SMs; integer sums, same frame).  Every eighth
            // pass is waited for, so that the progress line below stays within eight passes of the truth; checkpoints
            // and the download wait for everything by themselves.
            p.flags = (fresh ? 0 : (RT_FLAG_ACCUMULATE | RT_FLAG_ASYNC | RT_FLAG_OVERLAP)) | estimator_flags | (moments ? RT_FLAG_MOMENTS : 0u);
            fresh = false;
            if (rt_render(ctx, &p) != RT_OK) fail("rt_render");
            if (++passes % 8 == 0 && rt_sync(ctx) != RT_OK) fail("rt_sync");
            done += n;
            since_save += n;
            if (noise_target > 0 && done % check_every == 0 && done >= 2 && frame_noise() <= noise_target) {
                converged = true;
                std::cout << "\nNoise target " << noise_target << " reached at " << done << " samples per pixel" << std::endl;
            }
            if (!checkpoint_path.empty() && checkpoint_every_spp > 0 && since_save >= checkpoint_every_spp && done < samples_per_pixel && !converged) {
                save_checkpoint(done);
                since_save = 0;
            }
            std::cerr << "\rPercent Rendered: " << (100 * done / samples_per_pixel) << "% " << std::flush;
        }
        if (!checkpoint_path.empty()) {
            if (done < samples_per_pixel && !converged) save_checkpoint(done);  // stopped early: keep what we have
            else std::remove(checkpoint_path.c_str());              // finished: nothing left to resume
        }
        last_spp_done = done;
        last_rgb8.assign((size_t)p.width * p.height * 3, 0);
        const bool want_linear = !linear_name.empty();
        if (want_linear) last_linear.assign((size_t)p.width * p.height * 3, 0.0f);
        if (done > 0) {
            if (rt_download(ctx, done, want_linear ? last_linear.data() : nullptr, last_rgb8.data()) != RT_OK) fail("rt_download");
        }
        last_noise = moments && done >= 2 ? frame_noise() : 0.0;
        std::vector<float> variance;
        if (!variance_name.empty() && done >= 2) {
            variance.assign((size_t)p.width * p.height * 3, 0.0f);
            if (rt_download_variance(ctx, done, variance.data()) != RT_OK) fail("rt_download_variance");
        }
        rt_get_stats(ctx, &last_stats);
        rt_destroy(ctx);
        std::cout << "\nDone rendering " << image_name << std::endl;
        if (write_image) rtb200::write_png_rgb8(image_name, p.width, p.height, last_rgb8.data());
        if (want_linear) {
            const bool pfm = linear_name.size() >= 4 && linear_name.compare(linear_name.size() - 4, 4, ".pfm") == 0;
            bool ok = pfm ? rtb200::write_pfm(linear_name.c_str(), p.width, p.height, last_linear.data())
                          : rtb200::write_exr(linear_name.c_str(), p.width, p.height, last_linear.data());
            if (!ok) std::cerr << "rt_b200: cannot write " << linear_name << std::endl;
        }
        if (!variance.empty()) {
            const bool pfm = variance_name.size() >= 4 && variance_name.compare(variance_name.size() - 4, 4, ".pfm") == 0;
            bool ok = pfm ? rtb200::write_pfm(variance_name.c_str(), p.width, p.height, variance.data())
                          : rtb200::write_exr(variance_name.c_str(), p.width, p.height, variance.data());
            if (!ok) std::cerr << "rt_b200: cannot write " << variance_name << std::endl;
        }
    }

  private:
    // turntable_frames views of the uploaded scene in one batch (rt_render_views), progressive passes of up to 64
    // samples like render(); frame k is bit-identical to render() with turntable_camera(k)
    template <class Fail>
    void render_turntable(rt_ctx* ctx, Fail& fail) {
        const int n = turntable_frames, w = image_width, h = image_height();
        std::vector<rt_camera> cams((size_t)n);
        for (int k = 0; k < n; k++) cams[k] = turntable_camera(k);
        rt_render_params p;
        std::memset(&p, 0, sizeof p);
        p.struct_size = sizeof p;
        p.width = w;
        p.height = h;
        p.max_depth = max_depth;
        p.seed = seed;
        const uint32_t estimator_flags = (next_event_estimation ? RT_FLAG_NEE : 0u) | (shadowed_point_lights ? RT_FLAG_SHADOWED_POINT_LIGHTS : 0u);
        const int target = stop_after_spp > 0 ? std::min(stop_after_spp, samples_per_pixel) : samples_per_pixel;
        const int pass_spp = std::max(1, std::min(samples_per_pixel, 64));
        int done = 0, passes = 0;
        while (done < target) {
            const int k = std::min(pass_spp, target - done);
            p.samples_per_pixel = k;
            p.spp_begin = done;
            // passes after the first are enqueued without waiting; every eighth is waited for (the progress line)
            p.flags = (done == 0 ? 0u : (RT_FLAG_ACCUMULATE | RT_FLAG_ASYNC)) | estimator_flags;
            if (rt_render_views(ctx, &p, cams.data(), nullptr, n) != RT_OK) fail("rt_render_views");
            if (++passes % 8 == 0 && rt_sync(ctx) != RT_OK) fail("rt_sync");
            done += k;
            std::cerr << "\rPercent Rendered: " << (100 * done / samples_per_pixel) << "% " << std::flush;
        }
        last_spp_done = done;
        last_spp_resumed = 0;
        last_noise = 0;
        const size_t frame = (size_t)w * h * 3;
        last_rgb8.assign(frame * n, 0);
        const bool want_linear = !linear_name.empty();
        if (want_linear) last_linear.assign(frame * n, 0.0f);
        if (done > 0 && rt_download_views(ctx, done, 0, n, want_linear ? last_linear.data() : nullptr, last_rgb8.data()) != RT_OK)
            fail("rt_download_views");
        rt_get_stats(ctx, &last_stats);
        rt_destroy(ctx);
        std::cout << "\nDone rendering " << n << " turntable frames of " << image_name << std::endl;
        for (int k = 0; k < n; k++) {
            if (write_image) rtb200::write_png_rgb8(frame_name(image_name, k).c_str(), w, h, last_rgb8.data() + frame * k);
            if (want_linear) {
                const std::string name = frame_name(linear_name, k);
                const bool pfm = name.size() >= 4 && name.compare(name.size() - 4, 4, ".pfm") == 0;
                bool ok = pfm ? rtb200::write_pfm(name.c_str(), w, h, last_linear.data() + frame * k)
                              : rtb200::write_exr(name.c_str(), w, h, last_linear.data() + frame * k);
                if (!ok) std::cerr << "rt_b200: cannot write " << name << std::endl;
            }
        }
    }
};

#include "png_write.h"

#endif  // RTB200_RTOW_HOST_H
