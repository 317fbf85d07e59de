// area_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the spherical area lights of rm_render_area_lights (include/rm_b200.h,
// RmAreaLights) restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library
// unchanged).  direct_lighting and cast_ray (renderer.rs:138-309) are restated with the area term: a light of radius r > 0
// becomes s^2 point lights of colour k / s^2 on the disc that faces the shading point, each with the reference's own
// per-light term and shadow ray; the near-tie ("fragile") tracking of the oracle stays on.
#include "../oracle/rm_oracle.cpp"

namespace {

struct Area {
    const double* radius;     // one per light of the scene
    int s;
};

void lens_offset(int s, int i, int j, double& lx, double& ly) {
    const int a = (i + j) % s, b = j;
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    lx = p * std::sqrt(1. - (q * q) * 0.5);
    ly = q * std::sqrt(1. - (p * p) * 0.5);
}

// Duff et al. 2017, as the header states it
void light_frame(const V3 m, V3& t1, V3& t2) {
    const double sigma = std::copysign(1., m.z);
    const double alpha = -1. / (sigma + m.z);
    const double beta = (m.x * m.y) * alpha;
    t1 = V3{1. + ((sigma * m.x) * m.x) * alpha, sigma * beta, -sigma * m.x};
    t2 = V3{beta, sigma + (m.y * m.y) * alpha, -m.y};
}

V3 light_sample(const V3 c, const double r, const V3 t1, const V3 t2, const double lx, const double ly) {
    return V3{c.x + r * ((lx * t1.x) + (ly * t2.x)), c.y + r * ((lx * t1.y) + (ly * t2.y)), c.z + r * ((lx * t1.z) + (ly * t2.z))};
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
V3 area_direct(const V3& origin, const Hit& hit, const OrcScene& sc, const Area& A, Probe* pr) {
    V3 light_intensity{0, 0, 0};
    for (size_t l = 0; l < sc.lights.size(); l++) {
        const Light& light = sc.lights[l];
        const double r = A.radius[l];
        if (r == 0.) {
            point_term<T>(origin, hit, sc, light.position, light.color, light.intensity, light_intensity, pr);
            continue;
        }
        V3 t1, t2;
        light_frame(normalized(light.position - hit.point), t1, t2);
        const V3 color = scaled(light.color, 1. / (double)(A.s * A.s));
        for (int a = 0; a < A.s; a++)
            for (int b = 0; b < A.s; b++) {
                double lx, ly;
                lens_offset(A.s, a, b, lx, ly);
                point_term<T>(origin, hit, sc, light_sample(light.position, r, t1, t2, lx, ly), color, light.intensity, light_intensity, pr);
            }
    }
    return scaled(light_intensity, hit.refl.diffusion);                    // renderer.rs:192
}

// the oracle's cast_ray with area_direct in place of direct_lighting
template <bool T>
V3 cast_ray_area(const V3& orig, V3 dir, const OrcScene& sc, const Area& A, const V3& background, int n_recursion, int max_depth,
                 Probe* pr, int* primary_prim) {
    if (n_recursion > max_depth) return background;                        // renderer.rs:262-264
    Hit hit;
    if (T) pr->primary = (n_recursion == 1);
    bool got = find_closest_intersect<T>(orig, dir, sc, hit, pr);          // renderer.rs:266
    if (T) pr->primary = false;
    if (primary_prim) *primary_prim = got ? hit.prim : -1;
    if (!got) return (n_recursion > 1) ? background : V3{0, 0, 0};         // renderer.rs:300-306
    V3 light_intensity = background;                                       // renderer.rs:272
    light_intensity = light_intensity + area_direct<T>(orig, hit, sc, A, pr);   // renderer.rs:275
    if (hit.refl.is_glass_like) {                                          // renderer.rs:277
        V3 ro, rd;
        if (reflect_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr))
            light_intensity = light_intensity +
                scaled(cast_ray_area<T>(ro, rd, sc, A, background, n_recursion + 1, max_depth, pr, nullptr), hit.refl.reflection);
        if (refract_ray<T>(dir, hit, hit.refl.refractive_index, ro, rd, pr))
            light_intensity = light_intensity +
                scaled(cast_ray_area<T>(ro, rd, sc, A, background, n_recursion + 1, max_depth, pr, nullptr), 1. - hit.refl.reflection);
    }
    return light_intensity;
}

}  // namespace

extern "C" {

void orc_lens_offset_area(int s, int a, int b, double out[2]) { lens_offset(s, a, b, out[0], out[1]); }

void orc_light_frame(const double m[3], double t1[3], double t2[3]) {
    V3 a, b;
    light_frame(from3(m), a, b);
    to3(a, t1);
    to3(b, t2);
}

void orc_light_sample(const double c[3], double r, const double t1[3], const double t2[3], double lx, double ly, double q[3]) {
    to3(light_sample(from3(c), r, from3(t1), from3(t2), lx, ly), q);
}

// The area-light frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not
// written.  radius: one per light of the scene.  out_rgb H*W*3, prim_id H*W or null, fragile H*W or null (the oracle's bits).
int orc_render_area(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                    const double* radius, int n_radius, int s, double* out_rgb, int32_t* prim_id, uint8_t* fragile) {
    if (W <= 0 || H <= 0 || W % 32 != 0 || s < 1 || s > 8 || n_radius != (int)sc->lights.size()) return -1;
    const int n_height = H / 32;
    if (patch_row_end < 0 || patch_row_end > n_height) patch_row_end = n_height;
    if (patch_row_begin < 0) patch_row_begin = 0;
    const Area A{radius, s};
    const double half_fov = std::tan(fov / 2.);                            // renderer.rs:25-33
    const double height = (double)H, width = (double)W, ratio = width / height;
    const V3 background{0.1, 0.1, 0.1};                                    // renderer.rs:40-44
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
                const int i = next.fetch_add(1);
                if (i >= row_end) break;
                for (int j = 0; j < W; j++) {
                    // backproject(j, i), renderer.rs:128-135
                    V3 dir = normalized(V3{2. * ((double)j / width - 0.5) * half_fov * ratio, -2. * ((double)i / height - 0.5) * half_fov, -1.});
                    pr.fragile = 0;
                    int prim = -1;
                    const V3 c = cast_ray_area<true>(sc->camera, dir, *sc, A, background, 1, max_depth, &pr, &prim);
                    const size_t px = (size_t)i * W + j;
                    to3(c, out_rgb + 3 * px);
                    if (prim_id) prim_id[px] = prim;
                    if (fragile) fragile[px] = pr.fragile;
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    return 0;
}

}  // extern "C"
