// rough_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the rough glass of rm_render_rough_glass (include/rm_b200.h,
// RmRoughGlass) restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library
// unchanged, through tests/lens_oracle.cpp for the sample rays).  cast_ray (renderer.rs:254-309) is restated with the turn of
// every ray a rough glass-like hit spawns; the near-tie ("fragile") tracking of the oracle stays on, the side test of a
// turned ray's origin included.
#include "lens_oracle.cpp"

namespace {

struct Rough {
    const double* g;   // one per primitive id
    int n;
    int s, i, j;       // samples, and the sample being traced
};

// Duff et al. 2017, as the header states it
void rough_frame(const V3 m, V3& t1, V3& t2) {
    const double sigma = std::copysign(1., m.z);
    const double alpha = -1. / (sigma + m.z);
    const double beta = (m.x * m.y) * alpha;
    t1 = V3{1. + ((sigma * m.x) * m.x) * alpha, sigma * beta, -sigma * m.x};
    t2 = V3{beta, sigma + (m.y * m.y) * alpha, -m.y};
}

V3 rough_dir(const V3 rd, const double g, const double lx, const double ly) {
    if (!(g > 0.) || (lx == 0. && ly == 0.)) return rd;
    V3 t1, t2;
    rough_frame(rd, t1, t2);
    return normalized(V3{rd.x + g * ((lx * t1.x) + (ly * t2.x)), rd.y + g * ((lx * t1.y) + (ly * t2.y)),
                         rd.z + g * ((lx * t1.z) + (ly * t2.z))});
}

template <bool T>
V3 cast_ray_rough(const V3& orig, V3 dir, const OrcScene& sc, const Rough& R, const V3& background, int n_recursion, int max_depth,
                  Probe* pr, int* primary_prim) {
    if (n_recursion > max_depth) return background;                        // renderer.rs:262-264
    Hit hit;
    if (T) pr->primary = (n_recursion == 1);
    bool got = find_closest_intersect<T>(orig, dir, sc, hit, pr);          // renderer.rs:266
    if (T) pr->primary = false;
    if (primary_prim) *primary_prim = got ? hit.prim : -1;
    if (!got) return (n_recursion > 1) ? background : V3{0, 0, 0};         // renderer.rs:300-306
    V3 light_intensity = background;                                       // renderer.rs:272
    light_intensity = light_intensity + direct_lighting<T>(orig, hit, sc, pr);   // renderer.rs:275
    if (hit.refl.is_glass_like) {                                          // renderer.rs:277
        const double g = hit.prim >= 0 && hit.prim < R.n ? R.g[hit.prim] : 0.;
        double lx = 0., ly = 0.;
        lens_offset(R.s, (R.j + n_recursion) % R.s, R.i, lx, ly);        // stratum ((i + j + L) mod s, i)
        const bool turn = g > 0. && (lx != 0. || ly != 0.);
        V3 ro, rd;
        if (reflect_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr)) {
            if (turn) {
                rd = rough_dir(rd, g, lx, ly);
                const double side = dot(rd, hit.normal);
                if (T) pr->near(side, kF32);
                ro = side < 0. ? hit.point - scaled(hit.normal, 1e-4) : hit.point + scaled(hit.normal, 1e-4);
            }
            light_intensity = light_intensity +
                scaled(cast_ray_rough<T>(ro, rd, sc, R, background, n_recursion + 1, max_depth, pr, nullptr), hit.refl.reflection);
        }
        if (refract_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr)) {
            if (turn) {
                rd = rough_dir(rd, g, lx, ly);
                const V3 normal = -dot(hit.normal, dir) < 0. ? -hit.normal : hit.normal;
                const double side = dot(rd, normal);
                if (T) pr->near(side, kF32);
                ro = side > 0. ? hit.point + scaled(normal, 1e-4) : hit.point - scaled(normal, 1e-4);
            }
            light_intensity = light_intensity +
                scaled(cast_ray_rough<T>(ro, rd, sc, R, background, n_recursion + 1, max_depth, pr, nullptr), 1. - hit.refl.reflection);
        }
    }
    return light_intensity;
}

}  // namespace

extern "C" {

void orc_rough_dir(const double rd[3], double g, double lx, double ly, double out[3]) { to3(rough_dir(from3(rd), g, lx, ly), out); }

void orc_rough_offset(int s, int i, int j, int level, double out[2]) { lens_offset(s, (j + level) % s, i, out[0], out[1]); }

// The rough-glass frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not
// written.  roughness: n_rough values by primitive id.  out_rgb H*W*3: the f64 pixel means; frag_any H*W or null: the OR of
// a pixel's sample bits.
int orc_render_rough(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                     const double* basis, double aperture, double focus, int s, const double* roughness, int n_rough, double* out_rgb,
                     uint8_t* frag_any) {
    if (W <= 0 || H <= 0 || W % 32 != 0 || s < 1 || s > 8 || n_rough < 0) return -1;
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
                            const Rough R{roughness, n_rough, s, i, j};
                            const V3 c = cast_ray_rough<true>(o, d, *sc, R, background, 1, max_depth, &pr, nullptr);
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
