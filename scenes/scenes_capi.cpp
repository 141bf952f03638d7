// scenes_capi.cpp — builds the BASELINE scenes (scenes.h) against the host mirror of the
// reference's scene API and hands the flattened description to callers that are not C++
// (the pytest suite and bench.py, via ctypes).  Links against librt_b200.so because the
// mirror's camera::render calls the C ABI.
#ifdef RTB200_USE_STB_IMAGE
// JPEG / PNG textures decoded the way the reference decodes them: the user's own stb_image.h (the build adds the
// reference tree to the include path where it is mounted; stb_image is third-party I/O, outside the hot path)
#define STB_IMAGE_IMPLEMENTATION
#include "stb_image.h"
#endif
#include "rtow_host.h"

#include "scenes.h"

#include <chrono>

struct rtsc_scene {
    rtb200::flat_scene fs;
    rt_scene_desc desc;
    scene_config cfg;
    int max_depth;
};

extern "C" {

int rtsc_scene_count() {
    int n = 0;
    scene_names(&n);
    return n;
}
const char* rtsc_scene_name(int i) {
    int n = 0;
    const char* const* names = scene_names(&n);
    return (i >= 0 && i < n) ? names[i] : nullptr;
}

// mesh::indexed_meshes() for the scenes built from here on (rtsc_build, rtsc_render_png, rtsc_render_resumable):
// 1 loads their OBJ files as indexed meshes (rt_mesh), 0 (default) as triangle soups.  Returns the previous setting.
int rtsc_set_indexed_meshes(int on) {
    const bool was = mesh::indexed_meshes();
    mesh::indexed_meshes() = on != 0;
    return was ? 1 : 0;
}

// Builds scene `name` with construction seed `seed`; returns NULL for an unknown name.
rtsc_scene* rtsc_build(const char* name, unsigned seed, const char* asset_dir) {
    rtsc_scene* s = new rtsc_scene();
    if (asset_dir) s->cfg.asset_dir = asset_dir;
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!build_scene(name, seed, world, cam, lights, s->cfg)) {
        delete s;
        return nullptr;
    }
    rtb200::flatten_scene(world, lights, s->fs);
    cam.export_camera(s->fs.camera);
    s->desc = s->fs.desc();
    s->max_depth = cam.max_depth;
    return s;
}
const rt_scene_desc* rtsc_desc(const rtsc_scene* s) { return s ? &s->desc : nullptr; }
void rtsc_frame(const rtsc_scene* s, int* width, int* height, int* spp, int* depth) {
    if (width) *width = s->cfg.width;
    if (height) *height = s->cfg.height;
    if (spp) *spp = s->cfg.spp;
    if (depth) *depth = s->cfg.depth;
}
void rtsc_free(rtsc_scene* s) { delete s; }

// The whole reference-facing path in one call: build the scene with the mirror API and
// run camera::render (flatten -> rt_upload_scene -> rt_render -> rt_download -> PNG).
int rtsc_render_png(const char* name, unsigned seed, const char* asset_dir, int width, int height, int spp, int depth,
                    const char* out_png) {
    scene_config cfg;
    if (asset_dir) cfg.asset_dir = asset_dir;
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!build_scene(name, seed, world, cam, lights, cfg)) return 1;
    if (width > 0 && height > 0) { cam.image_width = width; cam.aspect_ratio = double(width) / double(height); }
    if (spp > 0) cam.samples_per_pixel = spp;
    if (depth > 0) cam.max_depth = depth;
    cam.image_name = out_png;
    cam.render(world, lights);
    return 0;
}

// The same call with the download-side additions (SURVEY 8f rank 3): a checkpoint file, an
// orderly stop after `stop_after_spp` samples, and a linear-radiance output (.exr / .pfm).
// Reports how many samples the frame holds and how many of them came from the checkpoint.
int rtsc_render_resumable(const char* name, unsigned seed, const char* asset_dir, int width, int height, int spp, int depth,
                          const char* out_png, const char* checkpoint, int checkpoint_every_spp, int stop_after_spp,
                          const char* linear_out, int* spp_done, int* spp_resumed) {
    scene_config cfg;
    if (asset_dir) cfg.asset_dir = asset_dir;
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!build_scene(name, seed, world, cam, lights, cfg)) return 1;
    if (width > 0 && height > 0) { cam.image_width = width; cam.aspect_ratio = double(width) / double(height); }
    if (spp > 0) cam.samples_per_pixel = spp;
    if (depth > 0) cam.max_depth = depth;
    cam.image_name = out_png;
    if (checkpoint) cam.checkpoint_path = checkpoint;
    cam.checkpoint_every_spp = checkpoint_every_spp;
    cam.stop_after_spp = stop_after_spp;
    if (linear_out) cam.linear_name = linear_out;
    cam.render(world, lights);
    if (spp_done) *spp_done = cam.last_spp_done;
    if (spp_resumed) *spp_resumed = cam.last_spp_resumed;
    return 0;
}

// camera::render as a turntable of `frames` views (camera::turntable_frames, one rt_render_views batch): frame k is
// written to <stem>_<k:03d><ext> of out_png.  nee / shadowed: the estimator flags.
int rtsc_render_turntable(const char* name, unsigned seed, const char* asset_dir, int width, int height, int spp, int depth,
                          const char* out_png, int frames, int nee, int shadowed) {
    scene_config cfg;
    if (asset_dir) cfg.asset_dir = asset_dir;
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!build_scene(name, seed, world, cam, lights, cfg)) return 1;
    if (width > 0 && height > 0) { cam.image_width = width; cam.aspect_ratio = double(width) / double(height); }
    if (spp > 0) cam.samples_per_pixel = spp;
    if (depth > 0) cam.max_depth = depth;
    cam.image_name = out_png;
    cam.turntable_frames = frames;
    cam.next_event_estimation = nee != 0;
    cam.shadowed_point_lights = shadowed != 0;
    cam.render(world, lights);
    return 0;
}

// The rt_camera of turntable frame k of `frames` for a BASELINE scene, as camera::turntable_camera computes it.
int rtsc_turntable_camera(const char* name, unsigned seed, const char* asset_dir, int frames, int k, rt_camera* out) {
    scene_config cfg;
    if (asset_dir) cfg.asset_dir = asset_dir;
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!out || !build_scene(name, seed, world, cam, lights, cfg)) return 1;
    cam.turntable_frames = frames;
    *out = cam.turntable_camera(k);
    return 0;
}

// mesh::loadObj on its own (SURVEY 8f rank 2).  loader = 1 selects the reference's structure
// (one shared_ptr<triangle> per face, mesh.h:22-121), 0 the fast path (parallel parse, one
// triangle_soup), 2 the fast path into one indexed_mesh (rt_mesh).  with_media adds three constant_medium spheres next to the mesh and wraps the list
// in a bvh_node, which makes the flattened media multiplicities depend on the replayed median split
// (Q15).  `ms` receives {load, bvh_node + flatten} in milliseconds.
rtsc_scene* rtsc_load_obj(const char* path, int loader, int with_media, float scale, double* ms) {
    using clk = std::chrono::steady_clock;
    rtsc_scene* s = new rtsc_scene();
    hittable_list world;
    auto mat = make_shared<lambertian>(color(0.5, 0.4, 0.3));
    mesh m;
    const bool saved = mesh::per_triangle_objects(), saved_indexed = mesh::indexed_meshes();
    mesh::per_triangle_objects() = loader == 1;
    mesh::indexed_meshes() = loader == 2;  // 0 is the soup, whatever rtsc_set_indexed_meshes says
    auto t0 = clk::now();
    glm::mat4 xf = glm::scale(glm::translate(glm::mat4(1.0f), glm::vec3(0.25f, -0.5f, 1.0f)), glm::vec3(scale));
    bool ok = m.loadObj(path, world, mat, xf);
    auto t1 = clk::now();
    mesh::per_triangle_objects() = saved;
    mesh::indexed_meshes() = saved_indexed;
    if (!ok) { delete s; return nullptr; }
    std::vector<point_light> lights;
    if (with_media) {
        world.add(make_shared<constant_medium>(make_shared<sphere>(point3(0, 0, 0), 0.3, mat), 0.5, color(1, 1, 1)));
        world.add(make_shared<constant_medium>(make_shared<sphere>(point3(40, 3, -20), 2.0, mat), 0.2, color(0, 0, 0)));
        world.add(make_shared<constant_medium>(make_shared<sphere>(point3(-1000, 0, 0), 5.0, mat), 0.1, color(0.2, 0.2, 0.2)));
        hittable_list wrapped(make_shared<bvh_node>(world));
        rtb200::flatten_scene(wrapped, lights, s->fs);
    } else {
        rtb200::flatten_scene(world, lights, s->fs);
    }
    auto t2 = clk::now();
    if (ms) {
        ms[0] = std::chrono::duration<double, std::milli>(t1 - t0).count();
        ms[1] = std::chrono::duration<double, std::milli>(t2 - t1).count();
    }
    camera cam;
    cam.lookfrom = point3(0, 2, 6);
    cam.lookat = point3(0, 0, 0);
    cam.background = color(0.7, 0.8, 1.0);
    cam.vfov = 40;
    cam.export_camera(s->fs.camera);
    s->desc = s->fs.desc();
    s->cfg.width = 320; s->cfg.height = 240; s->cfg.spp = 4; s->cfg.depth = 10;
    s->max_depth = 10;
    return s;
}

// The writers on their own (CPU tests): frame of w*h*3 floats -> file.
int rtsc_write_exr(const char* path, int w, int h, const float* rgb) { return rtb200::write_exr(path, w, h, rgb) ? 0 : 1; }
int rtsc_write_pfm(const char* path, int w, int h, const float* rgb) { return rtb200::write_pfm(path, w, h, rgb) ? 0 : 1; }
uint64_t rtsc_scene_hash(const rtsc_scene* s) { return s ? s->fs.hash() : 0; }
// 1 when this library decodes JPEG / PNG textures (built with the user's stb_image.h), 0 when only PPM / PGM
int rtsc_has_stb() {
#ifdef RTB200_USE_STB_IMAGE
    return 1;
#else
    return 0;
#endif
}

}  // extern "C"
