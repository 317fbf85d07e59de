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
        else if (a == "--samples") { need(1); samples = std::atoi(argv[++i]); }
        else if (a == "--contrast") { need(1); contrast = std::strtod(argv[++i], nullptr); adaptive = true; }
        else { std::fprintf(stderr, "rm_headless: unknown option %s\n", a.c_str()); return 2; }
    }
    if (samples < 1 || samples > 8 || ((samples > 1 || adaptive) && f64)) {
        std::fprintf(stderr, "rm_headless: --samples takes 1 to 8, with the FP32 kernels\n");
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

    RmParams p;
    rm_params_default(&p, width, height);                                  // fov 1.5 (main.rs:368), depth cap 3, background 0.1
    rm_builder_get_camera(b, p.camera);
    p.max_depth = depth;
    p.accel = accel;
    p.precision = f64 ? RM_FP64 : RM_FP32;
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
        if (f64) rc = rm_render_f64(scene, &p, rgb64.data(), nullptr, f == frames - 1 ? rgb8.data() : nullptr, &st);
        else if (rows64) rc = rm_render_rows_f64(scene, &p, row_ptrs.data(), RM_ROWS_RETAINED, &st);
        else rc = rm_render(scene, &p, rgb32.data(), nullptr, nullptr, &st);
        if (rc != RM_OK) die("render", rc);
        const long long ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        const double fps = 1000. / (double)ms;                             // renderer.rs:111-121 (0 ms prints inf, like the reference)
        std::printf("Scene rendered in %lld ms (%u fps, %.2f MP/s)\n", ms, ms > 0 ? (unsigned)fps : 4294967295u, fps * (double)n_px / 1e6);
    }
    // "Save to file": normalize + to_vec on the device (framebuffer.rs:40-82), then the P6 stream (framebuffer.rs:26-38)
    if (adaptive) {
        std::vector<unsigned char> mask(n_px, 0);
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render_adaptive(scene, &p, samples, contrast, nullptr, rgb8.data(), mask.data(), &st)) != RM_OK) die("render (adaptive 8-bit frame)", rc);
        size_t refined = 0;
        for (unsigned char m : mask) refined += m;
        std::printf("adaptive anti-aliasing: %zu of %zu pixels refined (%d x %d samples, contrast %g)\n", refined, n_px, samples, samples, contrast);
    } else if (samples > 1) {
        std::memset(&st, 0, sizeof st);
        if ((rc = rm_render_supersampled(scene, &p, samples, nullptr, rgb8.data(), &st)) != RM_OK) die("render (supersampled 8-bit frame)", rc);
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
