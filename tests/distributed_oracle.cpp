// distributed_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: distributed ray tracing of rm_render_distributed
// (include/rm_b200.h) restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library
// unchanged, through tests/motion_oracle.cpp for the scene at each sample's time and tests/lens_oracle.cpp for the sample
// rays).  cast_ray (renderer.rs:254-309) is restated with rough glass's turn and with rule 4's light point: a light of radius
// r > 0 is one point light of its full colour at the point of stratum area_offset(s, i, j, L) on the disc facing the shading
// point.  The near-tie ("fragile") tracking of the oracle stays on.
#include "motion_oracle.cpp"

namespace {

struct Dist {
    const double* radius;   // one per light of the scene, or null: every light a point
    const double* g;        // roughness by primitive id, or null
    int n_g;
    int s, i, j;            // samples, and the sample being traced
};

// Duff et al. 2017, as the header states it
void dist_frame(const V3 m, V3& t1, V3& t2) {
    const double sigma = std::copysign(1., m.z);
    const double alpha = -1. / (sigma + m.z);
    const double beta = (m.x * m.y) * alpha;
    t1 = V3{1. + ((sigma * m.x) * m.x) * alpha, sigma * beta, -sigma * m.x};
    t2 = V3{beta, sigma + (m.y * m.y) * alpha, -m.y};
}

V3 dist_rough_dir(const V3 rd, const double g, const double lx, const double ly) {
    if (!(g > 0.) || (lx == 0. && ly == 0.)) return rd;
    V3 t1, t2;
    dist_frame(rd, t1, t2);
    return normalized(V3{rd.x + g * ((lx * t1.x) + (ly * t2.x)), rd.y + g * ((lx * t1.y) + (ly * t2.y)),
                         rd.z + g * ((lx * t1.z) + (ly * t2.z))});
}

V3 dist_light_sample(const V3 c, const double r, const V3 t1, const V3 t2, const double lx, const double ly) {
    return V3{c.x + r * ((lx * t1.x) + (ly * t2.x)), c.y + r * ((lx * t1.y) + (ly * t2.y)), c.z + r * ((lx * t1.z) + (ly * t2.z))};
}

// rule 4: the stratum (a, b) = ((i + 2j + L) mod s, (i + 3j) mod s) taken to the unit disc by the elliptical grid map
void area_offset(const int s, const int i, const int j, const int level, double& lx, double& ly) {
    const int a = (i + 2 * j + level) % s, b = (i + 3 * j) % s;
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    lx = p * std::sqrt(1. - (q * q) * 0.5);
    ly = q * std::sqrt(1. - (p * p) * 0.5);
}

// one point light at `position` with `color`: the body of the oracle's direct_lighting loop (renderer.rs:166-189)
template <bool T>
void point_term(const V3& origin, const Hit& hit, const OrcScene& sc, const V3 position, const V3 color, const double intensity,
                V3& light_intensity, Probe* pr) {
    V3 light_dir = normalized(position - hit.point);                       // renderer.rs:166
    double side = dot(light_dir, hit.normal);
    if (T) {
        pr->c.light_evals++;
        double len = std::sqrt(squared_norm(position - hit.point));
        pr->near(side, kF32 * std::fmax(1., (max_abs3(position) + max_abs3(hit.point)) / std::fmax(len, 1e-300)));
    }
    V3 intersect_orig = (side < 0.) ? hit.point - scaled(hit.normal, 1e-3)    // renderer.rs:168-172
                                    : hit.point + scaled(hit.normal, 1e-3);
    if (intersect_shape_set<T>(intersect_orig, light_dir, sc, pr)) return;    // renderer.rs:174-177
    if (T) pr->c.lit_lights++;
    double diffusion = std::fmax(dot(light_dir, hit.normal), 0.);          // renderer.rs:138-140,180
    light_intensity = light_intensity + scaled(scaled(color * hit.refl.diffuse_color, diffusion), intensity);   // renderer.rs:181-183
    V3 incident = -light_dir;                                              // renderer.rs:144
    V3 reflected = reflect(incident, hit.normal);                          // renderer.rs:145
    V3 dir_to_viewer = normalized(origin - hit.point);                     // renderer.rs:149
    double spec_f = std::fmax(dot(reflected, dir_to_viewer), 0.);          // renderer.rs:150
    double specular = std::pow(spec_f * hit.refl.specular, hit.refl.specular_exponent);   // renderer.rs:186-188
    light_intensity = light_intensity + scaled(color, specular);           // renderer.rs:189
}

template <bool T>
V3 dist_direct(const V3& origin, const Hit& hit, const OrcScene& sc, const Dist& D, const int level, Probe* pr) {
    V3 light_intensity{0, 0, 0};
    for (size_t l = 0; l < sc.lights.size(); l++) {
        const Light& light = sc.lights[l];
        const double r = D.radius ? D.radius[l] : 0.;
        if (r == 0.) {
            point_term<T>(origin, hit, sc, light.position, light.color, light.intensity, light_intensity, pr);
            continue;
        }
        V3 t1, t2;
        dist_frame(normalized(light.position - hit.point), t1, t2);
        double lx, ly;
        area_offset(D.s, D.i, D.j, level, lx, ly);
        point_term<T>(origin, hit, sc, dist_light_sample(light.position, r, t1, t2, lx, ly), light.color, light.intensity, light_intensity, pr);
    }
    return scaled(light_intensity, hit.refl.diffusion);                    // renderer.rs:192
}

// the oracle's cast_ray with dist_direct in place of direct_lighting and rough glass's turn, in the scene `sc` (the scene
// at the sample's time)
template <bool T>
V3 cast_ray_dist(const V3& orig, V3 dir, const OrcScene& sc, const Dist& D, const V3& background, int n_recursion, int max_depth,
                 Probe* pr) {
    if (n_recursion > max_depth) return background;                        // renderer.rs:262-264
    Hit hit;
    if (T) pr->primary = (n_recursion == 1);
    bool got = find_closest_intersect<T>(orig, dir, sc, hit, pr);          // renderer.rs:266
    if (T) pr->primary = false;
    if (!got) return (n_recursion > 1) ? background : V3{0, 0, 0};         // renderer.rs:300-306
    V3 light_intensity = background;                                       // renderer.rs:272
    light_intensity = light_intensity + dist_direct<T>(orig, hit, sc, D, n_recursion, pr);   // renderer.rs:275
    if (hit.refl.is_glass_like) {                                          // renderer.rs:277
        const double g = D.g && hit.prim >= 0 && hit.prim < D.n_g ? D.g[hit.prim] : 0.;
        double lx = 0., ly = 0.;
        lens_offset(D.s, (D.j + n_recursion) % D.s, D.i, lx, ly);        // rough_offset: stratum ((i + j + L) mod s, i)
        const bool turn = g > 0. && (lx != 0. || ly != 0.);
        V3 ro, rd;
        if (reflect_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr)) {
            if (turn) {
                rd = dist_rough_dir(rd, g, lx, ly);
                const double side = dot(rd, hit.normal);
                if (T) pr->near(side, kF32);
                ro = side < 0. ? hit.point - scaled(hit.normal, 1e-4) : hit.point + scaled(hit.normal, 1e-4);
            }
            light_intensity = light_intensity +
                scaled(cast_ray_dist<T>(ro, rd, sc, D, background, n_recursion + 1, max_depth, pr), hit.refl.reflection);
        }
        if (refract_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr)) {
            if (turn) {
                rd = dist_rough_dir(rd, g, lx, ly);
                const V3 normal = -dot(hit.normal, dir) < 0. ? -hit.normal : hit.normal;
                const double side = dot(rd, normal);
                if (T) pr->near(side, kF32);
                ro = side > 0. ? hit.point + scaled(normal, 1e-4) : hit.point - scaled(normal, 1e-4);
            }
            light_intensity = light_intensity +
                scaled(cast_ray_dist<T>(ro, rd, sc, D, background, n_recursion + 1, max_depth, pr), 1. - hit.refl.reflection);
        }
    }
    return light_intensity;
}

}  // namespace

extern "C" {

void orc_area_offset(int s, int i, int j, int level, double out[2]) { area_offset(s, i, j, level, out[0], out[1]); }

// The distributed frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not
// written.  radius: n_radius values, one per light (null: point lights); roughness: n_rough values by primitive id (null:
// ideal optics); disp: 3 * n_disp values by primitive id (null: nothing moves).  out_rgb H*W*3: the f64 pixel means;
// frag_any H*W or null: the OR of a pixel's sample bits.
int orc_render_distributed(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin,
                           int patch_row_end, const double* basis, double aperture, double focus, int s, const double* radius, int n_radius,
                           const double* roughness, int n_rough, const double* disp, int n_disp, double* out_rgb, uint8_t* frag_any) {
    if (W <= 0 || H <= 0 || W % 32 != 0 || s < 1 || s > 8) return -1;
    if ((radius && n_radius != (int)sc->lights.size()) || (roughness && n_rough < 0) || (disp && n_disp != sc->n_prims)) return -1;
    const int n_height = H / 32;
    if (patch_row_end < 0 || patch_row_end > n_height) patch_row_end = n_height;
    if (patch_row_begin < 0) patch_row_begin = 0;
    const Lens L = make_lens(sc->camera, W, H, fov, basis, aperture, focus, s);
    const V3 background{0.1, 0.1, 0.1};                        // renderer.rs:40-44
    std::vector<OrcScene> at(disp ? (size_t)s * s : 0);        // the scene at the time of sample i s + j
    for (int i = 0; i < s && disp; i++)
        for (int j = 0; j < s; j++) scene_at(*sc, disp, motion_time(s, i, j), at[(size_t)i * s + j]);
    double scale = 1.;
    for (auto& sh : sc->shapes) scale = std::fmax(scale, sh->max_abs());
    for (const OrcScene& m : at)
        for (auto& sh : m.shapes) scale = std::fmax(scale, sh->max_abs());
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
                            const Dist D{radius, roughness, n_rough, s, i, j};
                            const OrcScene& scene = disp ? at[(size_t)i * s + j] : *sc;
                            const V3 c = cast_ray_dist<true>(o, d, scene, D, background, 1, max_depth, &pr);
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
