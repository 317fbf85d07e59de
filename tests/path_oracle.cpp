// path_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the path-traced frame of rm_render_path (include/rm_b200.h) restated
// over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library unchanged, through
// tests/distributed_oracle.cpp, which brings the scene at each sample's time, the sample rays, rough glass's turn and the area
// lights' one point per sample).  cast_ray (renderer.rs:254-309) is restated as distributed_oracle.cpp has it, with one diffuse
// ray per qualifying opaque hit as the header states rm_render_indirect's rule 2; the diffuse ray's hit is a shading point of
// level L + 1.  The near-tie ("fragile") tracking of the oracle stays on, the side test that turns the normal included.
#include "distributed_oracle.cpp"

namespace {

// the Shirley-Chiu concentric map of the centre of stratum (a, b), as the header states it
void path_diffuse_point(int s, int a, int b, double& lx, double& ly) {
    const double p = (2. * a + 1.) / s - 1., q = (2. * b + 1.) / s - 1.;
    const double pi = 3.14159265358979323846;
    if (p == 0. && q == 0.) {
        lx = 0.;
        ly = 0.;
        return;
    }
    double r, phi;
    if (std::fabs(p) > std::fabs(q)) {
        r = p;
        phi = (pi / 4.) * (q / p);
    } else {
        r = q;
        phi = pi / 2. - (pi / 4.) * (p / q);
    }
    lx = r * std::cos(phi);
    ly = r * std::sin(phi);
}

// the stratum ((2i + 3j + L) mod s, (3i + 5j) mod s)
void path_diffuse_offset(int s, int i, int j, int level, double& lx, double& ly) {
    path_diffuse_point(s, (2 * i + 3 * j + level) % s, (3 * i + 5 * j) % s, lx, ly);
}

// Malley's lift around n_f in the frame of rm::light_frame (dist_frame, Duff et al. 2017)
V3 path_diffuse_dir(const V3 nf, double lx, double ly) {
    V3 t1, t2;
    dist_frame(nf, t1, t2);
    const double z = std::sqrt(1. - ((lx * lx) + (ly * ly)));
    return normalized(V3{((lx * t1.x) + (ly * t2.x)) + z * nf.x, ((lx * t1.y) + (ly * t2.y)) + z * nf.y,
                         ((lx * t1.z) + (ly * t2.z)) + z * nf.z});
}

bool path_bounces(const Reflectance& r) {
    return !r.is_glass_like && r.diffusion > 0. && (r.diffuse_color.x > 0. || r.diffuse_color.y > 0. || r.diffuse_color.z > 0.);
}

// cast_ray_dist with the diffuse bounce, in the scene `sc` (the scene at the sample's time)
template <bool T>
V3 cast_ray_path(const V3& orig, V3 dir, const OrcScene& sc, const Dist& D, const V3& background, int n_recursion, int max_depth,
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
                scaled(cast_ray_path<T>(ro, rd, sc, D, background, n_recursion + 1, max_depth, pr), hit.refl.reflection);
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
                scaled(cast_ray_path<T>(ro, rd, sc, D, background, n_recursion + 1, max_depth, pr), 1. - hit.refl.reflection);
        }
    } else if (n_recursion < max_depth && path_bounces(hit.refl)) {
        double lx, ly;
        path_diffuse_offset(D.s, D.i, D.j, n_recursion, lx, ly);
        const double side = dot(hit.normal, dir);
        if (T) pr->near(side, kF32);
        const V3 nf = side < 0. ? hit.normal : -hit.normal;
        const V3 rd = path_diffuse_dir(nf, lx, ly);
        const V3 ro = hit.point + scaled(nf, 1e-4);
        const V3 v = cast_ray_path<T>(ro, rd, sc, D, background, n_recursion + 1, max_depth, pr);
        light_intensity = light_intensity + scaled(v * hit.refl.diffuse_color, hit.refl.diffusion);
    }
    return light_intensity;
}

}  // namespace

extern "C" {

// The path-traced frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not
// written.  radius: n_radius values, one per light (null: point lights); roughness: n_rough values by primitive id (null:
// ideal optics); disp: 3 * n_disp values by primitive id (null: nothing moves).  out_rgb H*W*3: the f64 pixel means;
// frag_any H*W or null: the OR of a pixel's sample bits.
int orc_render_path(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                    const double* basis, double aperture, double focus, int s, const double* radius, int n_radius, const double* roughness,
                    int n_rough, const double* disp, int n_disp, double* out_rgb, uint8_t* frag_any) {
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
                            const V3 c = cast_ray_path<true>(o, d, scene, D, background, 1, max_depth, &pr);
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
