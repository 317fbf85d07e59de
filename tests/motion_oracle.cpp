// motion_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the motion blur of rm_render_motion (include/rm_b200.h, RmMotion)
// restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library unchanged, through
// tests/lens_oracle.cpp for the sample rays).  For each of the s^2 sample times the scene's f64 geometry is moved to that
// time -- a sphere's centre, a polygon's vertices and plane point, a triangle's vertices and centre, each + tau*v, normals
// untouched -- and the sample is the oracle's own cast_ray in that scene, with the near-tie ("fragile") tracking on.
#include "lens_oracle.cpp"

#include <cstring>
#include <typeinfo>

namespace {

// the time of sample (i, j) of s x s, as the header states it
double motion_time(const int s, const int i, const int j) {
    const int m = s * ((2 * i + j) % s) + (i + j) % s;
    return ((double)m + 0.5) / (double)(s * s) - 0.5;
}

// p + tau*v component by component; a zero step (tau = 0 or v = 0) leaves p as it is
V3 moved(const V3 p, const double tau, const V3 v) {
    return {v.x != 0. && tau != 0. ? p.x + tau * v.x : p.x, v.y != 0. && tau != 0. ? p.y + tau * v.y : p.y,
            v.z != 0. && tau != 0. ? p.z + tau * v.z : p.z};
}

// The shapes come from the oracle library the caller built the scene with: its types are this file's by source but not by
// identity (anonymous namespace), so they are told apart by their type names.
template <class T> bool is_a(const Shape& s) { return std::strcmp(typeid(s).name(), typeid(T).name()) == 0; }

// the scene at time tau; disp: 3 values per primitive id
void scene_at(const OrcScene& sc, const double* disp, const double tau, OrcScene& out) {
    out.camera = sc.camera;
    out.lights = sc.lights;
    for (const auto& sh : sc.shapes) {
        const double* q = disp + 3 * (size_t)sh->prim_base;
        if (is_a<Sphere>(*sh)) {
            auto c = std::make_unique<Sphere>(static_cast<const Sphere&>(*sh));
            c->center = moved(c->center, tau, V3{q[0], q[1], q[2]});
            out.push(std::move(c));
        } else if (is_a<ConvexPolygon>(*sh)) {
            auto c = std::make_unique<ConvexPolygon>(static_cast<const ConvexPolygon&>(*sh));
            const V3 v{q[0], q[1], q[2]};
            for (auto& p : c->vertices) p = moved(p, tau, v);
            c->plane_point = moved(c->plane_point, tau, v);
            out.push(std::move(c));
        } else {
            auto c = std::make_unique<Obj>(static_cast<const Obj&>(*sh));
            for (size_t t = 0; t < c->triangles.size(); t++) {
                const V3 v{q[3 * t], q[3 * t + 1], q[3 * t + 2]};
                Triangle& tr = c->triangles[t];
                for (auto& p : tr.v) p = moved(p, tau, v);
                tr.center = moved(tr.center, tau, v);
            }
            out.push(std::move(c));
        }
    }
}

}  // namespace

extern "C" {

double orc_motion_time(int s, int i, int j) { return motion_time(s, i, j); }

// The motion frame over patch rows [patch_row_begin, patch_row_end) (end < 0: floor(H / 32)); rows outside are not written.
// disp: 3 * n_disp values by primitive id (n_disp must be the scene's primitive count).  out_rgb H*W*3: the f64 pixel means;
// frag_any H*W or null: the OR of a pixel's sample bits.
int orc_render_motion(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                      const double* basis, double aperture, double focus, int s, const double* disp, int n_disp, double* out_rgb,
                      uint8_t* frag_any) {
    if (W <= 0 || H <= 0 || W % 32 != 0 || s < 1 || s > 8 || n_disp != sc->n_prims) return -1;
    const int n_height = H / 32;
    if (patch_row_end < 0 || patch_row_end > n_height) patch_row_end = n_height;
    if (patch_row_begin < 0) patch_row_begin = 0;
    const Lens L = make_lens(sc->camera, W, H, fov, basis, aperture, focus, s);
    const V3 background{0.1, 0.1, 0.1};                        // renderer.rs:40-44
    std::vector<OrcScene> at((size_t)s * s);                   // the scene at the time of sample i s + j
    for (int i = 0; i < s; i++)
        for (int j = 0; j < s; j++) scene_at(*sc, disp, motion_time(s, i, j), at[(size_t)i * s + j]);
    double scale = 1.;
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
                            const V3 c = cast_ray<true>(o, d, at[(size_t)i * s + j], background, 1, max_depth, &pr, nullptr);
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
