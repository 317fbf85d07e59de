// view_oracle.cpp -- TEST INFRASTRUCTURE, never shipped: the camera orientation of rm_render_view (include/rm_b200.h,
// RmView) restated over the CPU oracle, which stays as it is (oracle/rm_oracle.cpp is compiled into this library
// unchanged).  The basis is built from the oracle's own geometry.rs restatement; the pixel loop is the oracle's
// render_patches with the definition applied to backproject's direction before cast_ray, so the near-tie ("fragile")
// mask follows the turned ray.
#include "../oracle/rm_oracle.cpp"

namespace {

template <bool T>
void render_patches_view(const OrcScene& sc, int W, int H, double fov, int max_depth, const V3 basis[3], const std::vector<int>& patches,
                         std::atomic<int>& next, double* out_rgb, int32_t* prim_id, uint8_t* fragile, Probe* pr) {
    const double half_fov = std::tan(fov / 2.);                 // renderer.rs:25-33
    const double height = (double)H, width = (double)W;
    const double ratio = width / height;
    const V3 background{0.1, 0.1, 0.1};                        // renderer.rs:40-44
    const int patch_size = 32;                                  // renderer.rs:47
    const int n_width = W / patch_size;
    const V3 u = basis[0], v = basis[1], w = basis[2];
    for (;;) {
        int k = next.fetch_add(1);
        if (k >= (int)patches.size()) break;
        int p = patches[k];
        int p_line = p % n_width * patch_size;                  // renderer.rs:69 (x)
        int p_col = p / n_width * patch_size;                   // renderer.rs:70 (y)
        for (int i = p_col; i < p_col + patch_size; i++) {
            for (int j = p_line; j < p_line + patch_size; j++) {
                // backproject(j, i), renderer.rs:128-135, then the view: ((u.x dx + v.x dy) + w.x dz, ...), not renormalised
                const V3 c0 = normalized(V3{2. * ((double)j / width - 0.5) * half_fov * ratio,
                                            -2. * ((double)i / height - 0.5) * half_fov, -1.});
                const V3 dir{(u.x * c0.x + v.x * c0.y) + w.x * c0.z, (u.y * c0.x + v.y * c0.y) + w.y * c0.z,
                             (u.z * c0.x + v.z * c0.y) + w.z * c0.z};
                int prim = -1;
                if (T) { pr->fragile = 0; pr->c.pixels++; }
                V3 c = cast_ray<T>(sc.camera, dir, sc, background, 1, max_depth, pr, &prim);
                size_t px = (size_t)i * W + j;                  // renderer.rs:92-108 reassembly
                out_rgb[3 * px] = c.x; out_rgb[3 * px + 1] = c.y; out_rgb[3 * px + 2] = c.z;
                if (prim_id) prim_id[px] = prim;
                if (T && fragile) fragile[px] = pr->fragile;
            }
        }
    }
}

}  // namespace

extern "C" {

// w = normalized(-forward), u = normalized(cross(up, w)), v = cross(w, u); -3 for an invalid view.
int orc_view_basis(const double forward[3], const double up_[3], double out[9]) {
    for (int a = 0; a < 3; a++)
        if (!std::isfinite(forward[a]) || !std::isfinite(up_[a])) return -3;
    const V3 f = from3(forward), up = from3(up_);
    if (dot(f, f) == 0.) return -3;
    const V3 w = normalized(-f);
    const V3 c = cross(up, w);
    if (dot(c, c) <= 1e-20 * dot(up, up)) return -3;
    const V3 u = normalized(c);
    to3(u, out);
    to3(cross(w, u), out + 3);
    to3(w, out + 6);
    return 0;
}

// orc_render with the primary rays turned by `basis` (u, v, w as orc_view_basis writes them).
int orc_render_view(const OrcScene* sc, int W, int H, double fov, int max_depth, int n_threads, int patch_row_begin, int patch_row_end,
                    int patch_stride, const double basis[9], double* out_rgb, int32_t* prim_id, uint8_t* fragile, OrcCounters* counters) {
    if (W <= 0 || H <= 0 || W % 32 != 0) return -1;
    const int n_height = H / 32, n_width = W / 32;
    if (patch_row_end < 0 || patch_row_end > n_height) patch_row_end = n_height;
    if (patch_row_begin < 0) patch_row_begin = 0;
    if (patch_stride < 1) patch_stride = 1;
    std::vector<int> patches;
    for (int p = patch_row_begin * n_width; p < patch_row_end * n_width; p += patch_stride) patches.push_back(p);
    if (n_threads < 1) n_threads = 1;
    const V3 b[3] = {from3(basis), from3(basis + 3), from3(basis + 6)};
    const bool track = prim_id || fragile || counters;
    double scale = 1.;
    for (auto& s : sc->shapes) scale = std::fmax(scale, s->max_abs());
    std::atomic<int> next{0};
    std::vector<Probe> probes(n_threads);
    for (auto& p : probes) p.scale = scale;
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) {
        Probe* pr = &probes[t];
        if (track)
            pool.emplace_back([&, pr] { render_patches_view<true>(*sc, W, H, fov, max_depth, b, patches, next, out_rgb, prim_id, fragile, pr); });
        else
            pool.emplace_back([&] { render_patches_view<false>(*sc, W, H, fov, max_depth, b, patches, next, out_rgb, nullptr, nullptr, nullptr); });
    }
    for (auto& th : pool) th.join();
    if (counters) {
        std::memset(counters, 0, sizeof(*counters));
        for (auto& p : probes) add_counters(*counters, p.c);
    }
    g_last_degenerate_hits = 0;
    for (auto& p : probes) g_last_degenerate_hits += p.degenerate_hits;
    return 0;
}

}  // extern "C"
