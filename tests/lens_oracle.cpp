// lens_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the thin-lens camera of rm_render_lens (include/rm_b200.h, RmLens)
// restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library unchanged).  The
// sample rays are built from the oracle's own geometry.rs restatement, each is traced by the oracle's cast_ray with the
// near-tie ("fragile") tracking on, and the pixel is the f64 mean of its samples in the normative order.
#include "../oracle/rm_oracle.cpp"

namespace {

struct Lens {
    double width, height, half_fov, ratio;      // of the s x frame
    V3 cam, u, v, w;
    double aperture, focus;
    int s;
};

void lens_offset(int s, int i, int j, double& lx, double& ly) {
    const int a = (i + j) % s, b = j;
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    lx = p * std::sqrt(1. - (q * q) * 0.5);
    ly = q * std::sqrt(1. - (p * p) * 0.5);
}

V3 world(const Lens& L, const V3 e) {
    return {(L.u.x * e.x + L.v.x * e.y) + L.w.x * e.z, (L.u.y * e.x + L.v.y * e.y) + L.w.y * e.z,
            (L.u.z * e.x + L.v.z * e.y) + L.w.z * e.z};
}

void lens_ray(const Lens& L, int x, int y, int i, int j, V3& o, V3& dir) {
    // backproject(s x + j, s y + i) of the s x frame, renderer.rs:128-135
    const V3 d = normalized(V3{2. * ((double)(L.s * x + j) / L.width - 0.5) * L.half_fov * L.ratio,
                               -2. * ((double)(L.s * y + i) / L.height - 0.5) * L.half_fov, -1.});
    if (L.aperture == 0.) {
        o = L.cam;
        dir = world(L, d);
        return;
    }
    double lx, ly;
    lens_offset(L.s, i, j, lx, ly);
    const double k = L.focus / (-d.z);
    const V3 P{d.x * k, d.y * k, d.z * k};
    const V3 Lp{L.aperture * lx, L.aperture * ly, 0.};
    const V3 e = normalized(P - Lp);
    o = V3{L.cam.x + (L.u.x * Lp.x + L.v.x * Lp.y), L.cam.y + (L.u.y * Lp.x + L.v.y * Lp.y), L.cam.z + (L.u.z * Lp.x + L.v.z * Lp.y)};
    dir = world(L, e);
}

Lens make_lens(const V3 cam, int W, int H, double fov, const double* basis, double aperture, double focus, int s) {
    Lens L;
    L.s = s;
    L.width = (double)(s * W);
    L.height = (double)(s * H);
    L.half_fov = std::tan(fov / 2.);                            // renderer.rs:25-33
    L.ratio = L.width / L.height;
    L.cam = cam;
    const double id[9] = {1., 0., 0., 0., 1., 0., 0., 0., 1.};
    const double* b = basis ? basis : id;
    L.u = from3(b);
    L.v = from3(b + 3);
    L.w = from3(b + 6);
    L.aperture = aperture;
    L.focus = focus;
    return L;
}

}  // namespace

extern "C" {

void orc_lens_offset(int s, int i, int j, double out[2]) { lens_offset(s, i, j, out[0], out[1]); }

// origin and direction of sample (i, j) of pixel (x, y) of a W x H frame; basis: u, v, w, or null for the reference's camera
void orc_lens_ray(const double cam[3], int W, int H, double fov, const double* basis, double aperture, double focus, int s, int x,
                  int y, int i, int j, double o[3], double d[3]) {
    const Lens L = make_lens(from3(cam), W, H, fov, basis, aperture, focus, s);
    V3 ro, rd;
    lens_ray(L, x, y, i, j, ro, rd);
    to3(ro, o);
    to3(rd, d);
}

// The lens frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not written.
//   out_rgb      H*W*3: the f64 pixel means
//   out_samples  H*W*s*s*3 or null: every sample value, sub-rows i outer, j inner
//   frag_samples H*W*s*s or null: the oracle's fragile bits of every sample ray
//   frag_any     H*W or null: the OR of a pixel's sample bits
int orc_render_lens(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                    const double* basis, double aperture, double focus, int s, double* out_rgb, double* out_samples,
                    uint8_t* frag_samples, uint8_t* frag_any) {
    if (W <= 0 || H <= 0 || W % 32 != 0 || s < 1 || s > 8) return -1;
    const int n_height = H / 32;
    if (patch_row_end < 0 || patch_row_end > n_height) patch_row_end = n_height;
    if (patch_row_begin < 0) patch_row_begin = 0;
    const Lens L = make_lens(sc->camera, W, H, fov, basis, aperture, focus, s);
    const V3 background{0.1, 0.1, 0.1};                        // renderer.rs:40-44
    double scale = 1.;
    for (auto& sh : sc->shapes) scale = std::fmax(scale, sh->max_abs());
    std::atomic<int> next{32 * patch_row_begin};
    const int row_end = 32 * patch_row_end;
    std::vector<std::thread> pool;
    if (n_threads < 1) n_threads = 1;
    for (int t = 0; t < n_threads; t++) {
        pool.emplace_back([&] {
            Probe pr;
            pr.scale = scale;
            for (;;) {
                const int y = next.fetch_add(1);
                if (y >= row_end) break;
                for (int x = 0; x < W; x++) {
                    const size_t px = (size_t)y * W + x;
                    V3 acc{0., 0., 0.};
                    uint8_t any = 0;
                    for (int i = 0; i < s; i++)
                        for (int j = 0; j < s; j++) {
                            V3 o, d;
                            lens_ray(L, x, y, i, j, o, d);
                            pr.fragile = 0;
                            int prim = -1;
                            const V3 c = cast_ray<true>(o, d, *sc, background, 1, max_depth, &pr, &prim);
                            const size_t k = px * s * s + (size_t)i * s + j;
                            if (out_samples) to3(c, out_samples + 3 * k);
                            if (frag_samples) frag_samples[k] = pr.fragile;
                            any |= pr.fragile;
                            acc = acc + c;
                        }
                    const double n = (double)(s * s);
                    to3(V3{acc.x / n, acc.y / n, acc.z / n}, out_rgb + 3 * px);
                    if (frag_any) frag_any[px] = any;
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    return 0;
}

}  // extern "C"
