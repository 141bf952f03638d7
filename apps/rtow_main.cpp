// rtow_main.cpp — what the reference's main.cpp (main.cpp:114-489) becomes on Linux with
// the B200 path underneath: the same include list, the same scene-construction code
// (scenes.h), the same `cam.render(world, lights)` call.  The Win32 shell glue of the
// reference (file dialogs, ShellExecuteW) is out of scope.
#ifdef RTB200_USE_STB_IMAGE
#define STB_IMAGE_IMPLEMENTATION
#include "stb_image.h"
#endif
#include "rtweekend.h"

#include "bvh.h"
#include "hittable_list.h"
#include "hittable.h"
#include "sphere.h"
#include "triangle.h"
#include "camera.h"
#include "quad.h"
#include "point_light.h"
#include "texture.h"
#include "constant_medium.h"
#include "mesh.h"

#include "scenes.h"

int main(int argc, char** argv) {
    std::string scene = argc > 1 ? argv[1] : "specular";  // main.cpp:120 defaults to scene 7
    std::string out = argc > 2 ? argv[2] : (scene + ".png");
    scene_config cfg;
    if (argc > 3) cfg.asset_dir = argv[3];
    hittable_list world;
    camera cam;
    std::vector<point_light> lights;
    if (!build_scene(scene, 1, world, cam, lights, cfg)) {
        std::cerr << "unknown scene " << scene << std::endl;
        return 1;
    }
    if (argc > 5) { cam.image_width = std::atoi(argv[4]); cam.aspect_ratio = double(cam.image_width) / std::atoi(argv[5]); }
    if (argc > 6) cam.samples_per_pixel = std::atoi(argv[6]);
    // additions: --checkpoint FILE [--every N] [--stop-after N] [--linear FILE.exr|.pfm] [--nee 0|1]
    //            --devices all | 0,1,2,...   split the frame over several GPUs of this box (one context, tiles gathered over NVLink)
    //            --noise X [--noise-every N]  stop once the relative frame noise is <= X, checked every N samples (default 256)
    //            --variance FILE.exr|.pfm     also write the per-pixel sample variance
    //            --turntable N                N views around lookat in one batch, written to <stem>_000<ext> ...
    for (int i = 7; i + 1 < argc; i += 2) {
        std::string k = argv[i];
        if (k == "--checkpoint") cam.checkpoint_path = argv[i + 1];
        else if (k == "--every") cam.checkpoint_every_spp = std::atoi(argv[i + 1]);
        else if (k == "--stop-after") cam.stop_after_spp = std::atoi(argv[i + 1]);
        else if (k == "--linear") cam.linear_name = argv[i + 1];
        else if (k == "--nee") cam.next_event_estimation = std::atoi(argv[i + 1]) != 0;
        else if (k == "--noise") cam.noise_target = std::atof(argv[i + 1]);
        else if (k == "--noise-every") cam.noise_check_every_spp = std::atoi(argv[i + 1]);
        else if (k == "--variance") cam.variance_name = argv[i + 1];
        else if (k == "--turntable") cam.turntable_frames = std::atoi(argv[i + 1]);
        else if (k == "--shadowed-point-lights") cam.shadowed_point_lights = std::atoi(argv[i + 1]) != 0;
        else if (k == "--devices") {
            std::string v = argv[i + 1];
            cam.devices.clear();
            if (v == "all") {
                int n = rt_visible_devices();
                for (int d = 0; d < n; d++) cam.devices.push_back(d);
            } else {
                size_t at = 0;
                while (at < v.size()) {
                    size_t c = v.find(',', at);
                    if (c == std::string::npos) c = v.size();
                    cam.devices.push_back(std::atoi(v.substr(at, c - at).c_str()));
                    at = c + 1;
                }
            }
        }
        else { std::cerr << "unknown option " << k << std::endl; return 1; }
    }
    cam.image_name = out.c_str();
    std::cout << "Rendering Image: " << cam.image_name << std::endl;
    cam.render(world, lights);
    if (cam.noise_target > 0 || !cam.variance_name.empty())
        std::cout << "Samples per pixel: " << cam.last_spp_done << ", relative noise " << cam.last_noise << std::endl;
    return 0;
}
