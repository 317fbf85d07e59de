// rm_headless.cpp -- a headless stand-in for the reference's GTK front end (engine/src/main.rs): what `cargo run` does when
// its buttons are pressed, driven through the C ABI only (include/rm_b200.h + rm_b200_host.h; no CUDA, no torch, no Python).
//
//   "Default scene"  main.rs:119-123  Scene::create_default          (no --obj)
//   "Open file"      main.rs:85-117,261-315  obj::load, every model moved by (0, 0, -500), the two lights    --obj FILE
//   camera buttons   main.rs:124-171  offset_camera(+-5 on an axis)   --camera X Y Z (accumulated offset)
//   render           main.rs:329-351  Renderer::render + the status label   (every run; --frames N re-renders N times,
//                                      the scene resident, like the re-render loop)
//   "Save to file"   main.rs:353-362  FrameBuffer::normalize + write_ppm("out.ppm")   --out FILE
//                                      --samples S (2..8): the saved frame anti-aliased, S x S primary rays per pixel
//                                      (rm_render_supersampled; an extension, the reference has no such mode)
//                                      --contrast C: S x S rays only where a pixel's 3x3 neighbourhood changes primitive
//                                      or exceeds the contrast C, one ray elsewhere (rm_render_adaptive; S = 1 without
//                                      --samples); prints the number of refined pixels
//   --look-at X,Y,Z                    the camera turned to look at that point (rm_render_view; an extension: the reference
//                                      always looks down -z), --up X,Y,Z its up direction (default 0,1,0).  Combines with
//                                      --camera, --accel, --f64 and --out; not with --samples, --contrast or --rows-f64
//   --aperture A --focus F             depth of field: a thin lens of radius A focused at distance F, --samples S x S rays
//                                      per pixel through it (rm_render_lens; an extension).  Combines with --samples,
//                                      --look-at / --up, --camera and --accel; not with --contrast, --f64 or --rows-f64
//   --light-radius R[,R...]            soft shadows: every light a sphere of radius R (one value for all lights, or one per
//                                      light in the scene's order), sampled at --samples S x S points of its disc
//                                      (rm_render_area_lights; an extension).  Combines with --samples, --camera and --accel;
//                                      not with --look-at, --aperture, --contrast, --f64 or --rows-f64
//   --roughness G                      rough glass: every ray a glass-like hit spawns turned within atan(G) of its ideal
//                                      direction, --samples S x S rays per pixel (rm_render_rough_glass; an extension; G for
//                                      every primitive).  Combines with --samples, --aperture / --focus, --look-at / --up,
//                                      --camera and --accel; not with --light-radius, --contrast, --f64 or --rows-f64
//   --move K,X,Y,Z                     motion blur: shape K of the scene (in scene order; every triangle of an Obj) moves by
//                                      (X, Y, Z) over the shutter, --samples S x S rays per pixel at S^2 times
//                                      (rm_render_motion; an extension).  Combines with --samples, --aperture / --focus,
//                                      --look-at / --up, --camera and --accel; not with --roughness, --light-radius,
//                                      --contrast, --f64 or --rows-f64
//   --combine                          distributed ray tracing: --light-radius, --roughness, --move, --aperture / --focus and
//                                      --look-at / --up all together, --samples S x S rays per pixel each sampling every
//                                      effect at once (rm_render_distributed; an extension; an area light is one point per
//                                      ray).  Not with --contrast, --f64 or --rows-f64
//   --indirect                         diffuse interreflection: every opaque hit spawns one cosine-weighted diffuse ray,
//                                      --samples S x S rays per pixel, --depth capping the whole path (rm_render_indirect;
//                                      an extension).  Combines with --samples, --aperture / --focus, --look-at / --up,
//                                      --camera and --accel; not with --light-radius, --roughness, --move, --combine,
//                                      --contrast, --f64 or --rows-f64
//   --path                             path-traced frames: --indirect's diffuse bounce with --combine's --light-radius,
//                                      --roughness, --move and --aperture / --focus, --samples S x S rays per pixel each
//                                      sampling every effect and every bounce at once, --depth capping the whole path
//                                      (rm_render_path; an extension).  Combines with --samples, --depth, --light-radius,
//                                      --roughness, --move, --aperture / --focus, --look-at / --up, --camera and --accel; not
//                                      with --combine, --indirect, --contrast, --f64 or --rows-f64
//
//   g++ -std=c++17 -Iinclude examples/rm_headless.cpp -o examples/rm_headless -Lrusty_marcher_b200 -lrm_b200 -Wl,-rpath,'$ORIGIN/../rusty_marcher_b200'
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rm_b200.h"
#include "rm_b200_host.h"

static void die(const char* what, int rc) {
    std::fprintf(stderr, "rm_headless: %s failed (%d): %s\n", what, rc, rm_last_error());
    std::exit(1);
}

int main(int argc, char** argv) {
    int width = 1600, height = 1280, depth = 3, frames = 1, accel = 0, samples = 1;     // main.rs:240: the frame buffer is 1600 x 1280
    bool f64 = false, rows64 = false;
    const char* obj = nullptr;
    const char* out = "out.ppm";
    bool adaptive = false;
    double contrast = 0.;
    double cam[3] = {0., 0., 0.};
    bool look = false;
    double target[3] = {0., 0., 0.};
    RmView view = {{0., 0., -1.}, {0., 1., 0.}};
    bool use_lens = false, have_focus = false;
    RmLens lens = {0., 1., 1};
    bool area = false;
    std::vector<double> radii;
    bool rough = false;
    double roughness = 0.;
    bool moving = false;
    bool combine = false;
    bool indirect = false;
    bool path = false;
    int move_shape = -1;
    double move_by[3] = {0., 0., 0.};
    auto triple = [](const char* s, double v[3]) { char end = 0; return std::sscanf(s, "%lf,%lf,%lf%c", &v[0], &v[1], &v[2], &end) == 3; };
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto need = [&](int n) { if (i + n >= argc) { std::fprintf(stderr, "rm_headless: %s needs %d value(s)\n", a.c_str(), n); std::exit(2); } };
        if (a == "--obj") { need(1); obj = argv[++i]; }
        else if (a == "--width") { need(1); width = std::atoi(argv[++i]); }
        else if (a == "--height") { need(1); height = std::atoi(argv[++i]); }
        else if (a == "--depth") { need(1); depth = std::atoi(argv[++i]); }
        else if (a == "--frames") { need(1); frames = std::atoi(argv[++i]); }
        else if (a == "--camera") { need(3); for (int k = 0; k < 3; k++) cam[k] = std::atof(argv[++i]); }
        else if (a == "--out") { need(1); out = argv[++i]; }
        else if (a == "--f64") f64 = true;              // the validation kernels: the reference's own f64 arithmetic
        else if (a == "--rows-f64") rows64 = true;      // FP32 kernels into the reference's frame type (one allocation per row, f64)
        else if (a == "--accel") accel = 1;
        else if (a == "--combine") combine = true;
        else if (a == "--indirect") indirect = true;
        else if (a == "--path") path = true;
        else if (a == "--samples") { need(1); samples = std::atoi(argv[++i]); }
        else if (a == "--contrast") { need(1); contrast = std::strtod(argv[++i], nullptr); adaptive = true; }
        else if (a == "--aperture") { need(1); lens.aperture = std::strtod(argv[++i], nullptr); use_lens = true; }
        else if (a == "--focus") { need(1); lens.focus = std::strtod(argv[++i], nullptr); have_focus = true; }
        else if (a == "--roughness") { need(1); roughness = std::strtod(argv[++i], nullptr); rough = true; }
        else if (a == "--move") {
            need(1);
            char end = 0;
            if (std::sscanf(argv[++i], "%d,%lf,%lf,%lf%c", &move_shape, &move_by[0], &move_by[1], &move_by[2], &end) != 4) {
                std::fprintf(stderr, "rm_headless: --move takes K,X,Y,Z\n");
                return 2;
            }
            moving = true;
        }
        else if (a == "--light-radius") {
            need(1);
            area = true;
            radii.clear();
            for (const char* q = argv[++i];;) {
                char* end = nullptr;
                radii.push_back(std::strtod(q, &end));
                if (end == q || (*end != ',' && *end != 0)) { std::fprintf(stderr, "rm_headless: --light-radius takes R[,R...]\n"); return 2; }
                if (*end == 0) break;
                q = end + 1;
            }
        }
        else if (a == "--look-at" || a == "--up") {
            need(1);
            if (!triple(argv[++i], a == "--up" ? view.up : target)) { std::fprintf(stderr, "rm_headless: %s takes X,Y,Z\n", a.c_str()); return 2; }
            look = look || a == "--look-at";
        }
        else { std::fprintf(stderr, "rm_headless: unknown option %s\n", a.c_str()); return 2; }
    }
    if (samples < 1 || samples > 8 || ((samples > 1 || adaptive) && f64)) {
        std::fprintf(stderr, "rm_headless: --samples takes 1 to 8, with the FP32 kernels\n");
        return 2;
    }
    if (use_lens != have_focus || (use_lens && (adaptive || f64 || rows64))) {
        std::fprintf(stderr, "rm_headless: --aperture and --focus go together, and not with --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    lens.samples = samples;
    if (combine && (adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --combine does not combine with --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (path && (combine || indirect || adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --path does not combine with --combine, --indirect, --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (indirect && (area || rough || moving || combine || adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --indirect does not combine with --light-radius, --roughness, --move, --combine, --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (area && !combine && !path && (look || use_lens || adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --light-radius does not combine with --look-at, --aperture, --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (rough && !combine && !path && (area || adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --roughness does not combine with --light-radius, --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (moving && !combine && !path && (rough || area || adaptive || f64 || rows64)) {
        std::fprintf(stderr, "rm_headless: --move does not combine with --roughness, --light-radius, --contrast, --f64 or --rows-f64\n");
        return 2;
    }
    if (look && !combine && !path && !indirect && !use_lens && !rough && !moving && (samples > 1 || adaptive || rows64)) {
        std::fprintf(stderr, "rm_headless: --look-at does not combine with --samples, --contrast or --rows-f64\n");
        return 2;
    }
    if (contrast != contrast) {
        std::fprintf(stderr, "rm_headless: --contrast takes a number (not NaN)\n");
        return 2;
    }
    int rc = rm_init(0);
    if (rc != RM_OK) die("rm_init", rc);

    RmSceneBuilder* b = nullptr;
    if (obj) {
        b = rm_builder_new();
        const double offset[3] = {0., 0., -500.};                          // main.rs:278-282
        const int n = rm_builder_add_obj_file(b, obj, offset);
        if (n < 0) { std::printf("Could not load obj from %s\n", obj); return 1; }      // obj.rs:53-56
        const double l0[3] = {0., 0., 0.}, c0[3] = {1., 1., 1.}, l1[3] = {20., 20., 20.}, c1[3] = {1., .5, .5};
        rm_builder_add_light(b, l0, c0, 1.);                               // main.rs:293-315
        rm_builder_add_light(b, l1, c1, .8);
    } else {
        b = rm_builder_create_default();                                   // scene.rs:28-211
    }
    rm_builder_offset_camera(b, cam);
    RmScene scene = 0;
    if ((rc = rm_builder_upload(b, &scene)) != RM_OK) die("rm_scene_upload", rc);

    RmAreaLights area_lights = {0, nullptr, samples};
    if (area) {
        const int n_lights = rm_builder_flatten(b)->n_lights;
        if (radii.size() == 1) radii.assign(n_lights, radii[0]);
        if ((int)radii.size() != n_lights) {
            std::fprintf(stderr, "rm_headless: --light-radius takes one radius or %d (one per light)\n", n_lights);
            return 2;
        }
        area_lights.n_lights = n_lights;
        area_lights.radius = radii.data();
    }

    std::vector<double> rough_g;
    RmRoughGlass rough_glass = {0, nullptr, samples};
    if (rough) {
        rough_g.assign(rm_scene_num_prims(scene), roughness);
        rough_glass.n_prims = (int)rough_g.size();
        rough_glass.roughness = rough_g.data();
    }

    std::vector<double> disp;
    RmMotion motion = {0, nullptr, samples};
    if (moving) {
        const RmFlatScene* fs = rm_builder_flatten(b);
        if (move_shape < 0 || move_shape >= fs->n_shapes) {
            std::fprintf(stderr, "rm_headless: --move: the scene has shapes 0 to %d\n", fs->n_shapes - 1);
            return 2;
        }
        disp.assign(3 * (size_t)rm_scene_num_prims(scene), 0.);
        size_t first = 0;                                                  // primitive ids: shapes in order, an Obj per triangle
        for (int k = 0; k <= move_shape; k++) {
            const int n = fs->shapes[k].kind == RM_SHAPE_OBJ ? fs->objs[fs->shapes[k].index].n_triangles : 1;
            if (k == move_shape)
                for (int t = 0; t < n; t++)
                    for (int c = 0; c < 3; c++) disp[3 * (first + t) + c] = move_by[c];
            first += n;
        }
        motion.n_prims = rm_scene_num_prims(scene);
        motion.displacement = disp.data();
    }

    RmParams p;
    rm_params_default(&p, width, height);                                  // fov 1.5 (main.rs:368), depth cap 3, background 0.1
    rm_builder_get_camera(b, p.camera);
    p.max_depth = depth;
    p.accel = accel;
    p.precision = f64 ? RM_FP64 : RM_FP32;
    if (look) {
        for (int k = 0; k < 3; k++) view.forward[k] = target[k] - p.camera[k];
        double basis[9];
        if ((rc = rm_view_basis(&view, basis)) != RM_OK) {
            std::fprintf(stderr, "rm_headless: %s\n", rm_last_error());
            return 2;
        }
    }
    const size_t n_px = (size_t)width * height;
    std::vector<unsigned char> rgb8(n_px * 3, 0);
    std::vector<float> rgb32;
    std::vector<double> rgb64;
    std::vector<std::vector<double>> frame_rows;                           // framebuffer.rs:6-10: Vec<Vec<Vec3f>>
    std::vector<double*> row_ptrs;
    if (f64) rgb64.assign(n_px * 3, 0.);
    else if (rows64) {
        frame_rows.assign(height, std::vector<double>((size_t)width * 3, 0.));
        for (auto& r : frame_rows) row_ptrs.push_back(r.data());
    } else rgb32.assign(n_px * 3, 0.f);

    if (height % 32 != 0 || width % 32 != 0) std::printf("Dimensions mismatch\n");                       // renderer.rs:49-51
    std::printf("Rendering using patches of size %d, using %d patches overall\n", 32, (height / 32) * (width / 32));
    RmStats st;
    for (int f = 0; f < frames; f++) {
        const auto t0 = std::chrono::steady_clock::now();
        std::memset(&st, 0, sizeof st);
        if (path) rc = rm_render_path(scene, &p, samples, look ? &view : nullptr, use_lens ? &lens : nullptr, area ? &area_lights : nullptr,
                                      rough ? &rough_glass : nullptr, moving ? &motion : nullptr, rgb32.data(),
                                      f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (combine) rc = rm_render_distributed(scene, &p, samples, look ? &view : nullptr, use_lens ? &lens : nullptr, area ? &area_lights : nullptr,
                                                rough ? &rough_glass : nullptr, moving ? &motion : nullptr, rgb32.data(),
                                                f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (indirect) rc = rm_render_indirect(scene, &p, look ? &view : nullptr, use_lens ? &lens : nullptr, samples, rgb32.data(),
                                                   f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (moving) rc = rm_render_motion(scene, &p, look ? &view : nullptr, use_lens ? &lens : nullptr, &motion, rgb32.data(),
                                          f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (rough) rc = rm_render_rough_glass(scene, &p, look ? &view : nullptr, use_lens ? &lens : nullptr, &rough_glass, rgb32.data(),
                                              f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (area) rc = rm_render_area_lights(scene, &p, &area_lights, rgb32.data(), nullptr, f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (use_lens) rc = rm_render_lens(scene, &p, look ? &view : nullptr, &lens, rgb32.data(), f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (look && f64) rc = rm_render_view_f64(scene, &p, &view, rgb64.data(), nullptr, f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (look) rc = rm_render_view(scene, &p, &view, rgb32.data(), nullptr, nullptr, &st);
        else if (f64) rc = rm_render_f64(scene, &p, rgb64.data(), nullptr, f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (rows64) rc = rm_render_rows_f64(scene, &p, row_ptrs.data(), RM_ROWS_RETAINED, &st);
        else rc = rm_render(scene, &p, rgb32.data(), nullptr, nullptr, &st);
        if (rc != RM_OK) die("render", rc);
        const long long ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        const double fps = 1000. / (double)ms;                             // renderer.rs:111-121 (0 ms prints inf, like the reference)
        std::printf("Scene rendered in %lld ms (%u fps, %.2f MP/s)\n", ms, ms > 0 ? (unsigned)fps : 4294967295u, fps * (double)n_px / 1e6);
    }
    // "Save to file": normalize + to_vec on the device (framebuffer.rs:40-82), then the P6 stream (framebuffer.rs:26-38)
    if (path || combine || indirect || use_lens || area || rough || moving) {
        // (the last frame above wrote the 8-bit frame)
    } else if (adaptive) {
        std::vector<unsigned char> mask(n_px, 0);
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render_adaptive(scene, &p, samples, contrast, nullptr, rgb8.data(), mask.data(), &st)) != RM_OK) die("render (adaptive 8-bit frame)", rc);
        size_t refined = 0;
        for (unsigned char m : mask) refined += m;
        std::printf("adaptive anti-aliasing: %zu of %zu pixels refined (%d x %d samples, contrast %g)\n", refined, n_px, samples, samples, contrast);
    } else if (samples > 1) {
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render_supersampled(scene, &p, samples, nullptr, rgb8.data(), &st)) != RM_OK) die("render (supersampled 8-bit frame)", rc);
    } else if (look && !f64) {
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render_view(scene, &p, &view, nullptr, nullptr, rgb8.data(), &st)) != RM_OK) die("render (8-bit frame)", rc);
    } else if (!f64) {
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render(scene, &p, nullptr, nullptr, rgb8.data(), &st)) != RM_OK) die("render (8-bit frame)", rc);
    }
    if ((rc = rm_write_ppm(out, width, height, rgb8.data())) != RM_OK) die("rm_write_ppm", rc);
    std::printf("max %.17g, %d primitives resident, saved %s\n", st.max_value, st.resident_prims, out);
    rm_scene_free(scene);
    rm_builder_free(b);
    rm_shutdown();
    return 0;
}
