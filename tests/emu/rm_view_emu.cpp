// rm_view_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// The camera orientation of rm_render_view through the product's own kernel code compiled for the host, next to
// rm_emu.cpp's emu_render_fast / emu_render_f64 (included here unchanged): K0's rotated raster records (prepare_raster with
// the basis), stage A on them with the warp strips' exact bound and the classify kernel's tile bound, or the hierarchy,
// and the shading stage with the turned primary directions -- and the generic kernel's FP64 path with the definition
// applied to backproject.
#include "rm_emu.cpp"

namespace {

rm::ViewBasis view_basis_of(const double basis[9]) {
    rm::ViewBasis vb;
    for (int k = 0; k < 9; k++) {
        vb.m[k] = basis[k];
        vb.f[k] = (float)basis[k];
    }
    return vb;
}

template <bool kBvh>
int emu_render_fast_view_impl(const RmFlatScene* fs, const RmParams* p, const rm::ViewBasis& vw, float* out_rgb, int32_t* prim,
                              int n_threads) {
    rm::PackedScene<float> ps;
    std::string err;
    int rc = rm::pack_scene<float>(*fs, ps, err);
    if (rc != RM_OK) return rc;
    if (p->width % 32) return RM_ERR_DIMENSIONS;
    const bool cull = p->cull_backfacing != 0;
    const rm::BlobLayout& L = ps.lay;
    const unsigned char* base = ps.blob_data();
    const int n_tri = rm::tri_count(L, cull);
    std::vector<rm::R4<float>> tri_r((size_t)n_tri * 4 + 4);
    for (int j = 0; j < n_tri; j++) rm::prepare_raster(ps.tri_src.data() + (size_t)j * rm::kTriSrcDoubles, p->camera, tri_r.data() + 4 * j, vw);
    rm::FastViewT<kBvh> fv0;
    fv0.bvh.nodes = ps.bvh_nodes.data();
    fv0.bvh.prims = ps.bvh_prims.data();
    fv0.bvh.n_nodes = (int)(ps.bvh_nodes.size() / 4);
    fv0.sph = reinterpret_cast<const rm::R4<float>*>(base + L.off_sph);
    fv0.sph_id = reinterpret_cast<const int*>(base + L.off_sph_id);
    fv0.n_sph = L.n_sph;
    fv0.tri_g = reinterpret_cast<const rm::R4<float>*>(base + L.off_tri_g);
    fv0.tri_r = tri_r.data();
    fv0.n_tri = n_tri;
    fv0.poly_slot = reinterpret_cast<const int*>(base + L.off_poly_slot);
    fv0.n_poly = rm::poly_count(L, cull);
    fv0.pln_n = reinterpret_cast<const rm::R4<float>*>(base + L.off_pln_n);
    fv0.pln_c = reinterpret_cast<const rm::R4<float>*>(base + L.off_pln_c);
    fv0.pln_v = reinterpret_cast<const rm::I2*>(base + L.off_pln_v);
    fv0.pln_id = reinterpret_cast<const int*>(base + L.off_pln_id);
    fv0.vert = reinterpret_cast<const rm::R4<float>*>(base + L.off_vert);
    fv0.mat_a = ps.mat_a.data();
    fv0.mat_b = ps.mat_b.data();
    fv0.mat_f = ps.mat_f.data();
    fv0.lgt_p = reinterpret_cast<const rm::R4<float>*>(base + L.off_lgt_p);
    fv0.lgt_c = reinterpret_cast<const rm::R4<float>*>(base + L.off_lgt_c);
    fv0.n_lgt = L.n_lgt;
    fv0.sph64 = ps.sph64.data();
    fv0.tri64 = ps.tri_src.data();
    fv0.pln64 = ps.pln64.data();
    const rm::FrameParams<float> fp = rm::make_frame_params<float>(*p);
    const int gm = g_glass_mode.load() >= 0 ? g_glass_mode.load() : rm::glass_mode(L.any_glass != 0, L.n_sph, L.coord_max, L.r_min, p->camera);
    g_last_glass_mode.store(gm);
    const bool bound = g_strip_bound.load() != 0;
    std::atomic<int> next{fp.row_begin};
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) {
        pool.emplace_back([&] {
            rm::FastViewT<kBvh> fv = fv0;
            std::vector<int> cand;
            for (;;) {
                const int y0 = next.fetch_add(4);
                if (y0 >= fp.row_end) break;
                for (int xs = 0; xs < fp.width; xs += 32) {
                    const float Xa = rm::pixel_X(fp, xs), Xb = rm::pixel_X(fp, xs + 31);
                    const float Ya = rm::pixel_Y(fp, y0), Yb = rm::pixel_Y(fp, y0 + 3);
                    // the classify kernel's tile bound on the rotated records: provably empty tiles are only zero-filled
                    bool tile_busy = kBvh || fv.n_sph + fv.n_poly > 0 || !bound;
                    const int ty0 = fp.row_begin + ((y0 - fp.row_begin) / 32) * 32;
                    const float TYa = rm::pixel_Y(fp, ty0), TYb = rm::pixel_Y(fp, ty0 + 31);
                    for (int j = 0; j < n_tri && !tile_busy; j++)
                        tile_busy = rm::tri_may_touch(tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], Xa, Xb, TYa, TYb);
                    if (!tile_busy) {
                        for (int y = y0; y < y0 + 4; y++)
                            for (int x = xs; x < xs + 32; x++) {
                                const size_t px = (size_t)y * fp.width + x;
                                out_rgb[3 * px] = out_rgb[3 * px + 1] = out_rgb[3 * px + 2] = 0.f;
                                if (prim) prim[px] = -1;
                            }
                        continue;
                    }
                    cand.clear();
                    for (int j = 0; j < n_tri && !kBvh; j++)
                        if (!bound || rm::tri_may_touch(tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], Xa, Xb, Ya, Yb)) cand.push_back(j);
                    for (int lane = 0; lane < 32; lane++) {
                        const int x = xs + (lane & 7) * 4, y = y0 + (lane >> 3);
                        rm::PrimaryState<4> st;
                        rm::primary_begin<4>(st, fp, x, y);
                        if constexpr (kBvh) {
                            rm::primary_bvh<4>(st, fv, fp, vw);
                        } else {
                            for (int j : cand) rm::primary_tri<4>(st, tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], fv.n_sph + j);
                            if (fv.n_sph + fv.n_poly > 0) rm::primary_rest<4>(st, fv, fp, vw);
                        }
                        for (int k = 0; k < 4; k++) {
                            rm::Vec3<float> c = {0.f, 0.f, 0.f};
                            if (st.slot[k] >= 0)
                                c = gm == rm::GLASS_NONE  ? rm::fast_shade<rm::GLASS_NONE>(fv, fp, x + k, y, st.t[k], st.slot[k], st.id[k], vw)
                                    : gm == rm::GLASS_F32 ? rm::fast_shade<rm::GLASS_F32>(fv, fp, x + k, y, st.t[k], st.slot[k], st.id[k], vw)
                                                          : rm::fast_shade<rm::GLASS_F64>(fv, fp, x + k, y, st.t[k], st.slot[k], st.id[k], vw);
                            const size_t px = (size_t)y * fp.width + x + k;
                            out_rgb[3 * px] = c.x; out_rgb[3 * px + 1] = c.y; out_rgb[3 * px + 2] = c.z;
                            if (prim) prim[px] = st.id[k];
                        }
                    }
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    return RM_OK;
}

// the generic kernel's loop (render_kernel<R, S, kView>): cast_ray from view.apply(backproject(x, y)), counters on
template <typename R>
int emu_render_view_impl(const RmFlatScene* fs, const RmParams* p, const rm::ViewBasis& vw, R* out_rgb, int32_t* prim, RmStats* stats,
                         int n_threads) {
    rm::PackedScene<R> ps;
    std::string err;
    int rc = rm::pack_scene<R>(*fs, ps, err);
    if (rc != RM_OK) return rc;
    if (p->width % 32) return RM_ERR_DIMENSIONS;
    const rm::SceneView<R> sc = view_of(ps, p->cull_backfacing != 0);
    const rm::FrameParams<R> fp = rm::make_frame_params<R>(*p);
    std::atomic<int> next{fp.row_begin};
    std::vector<rm::Counters<true>> tc(n_threads);
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) {
        pool.emplace_back([&, t] {
            rm::Counters<true>& st = tc[t];
            st.clear();
            for (;;) {
                const int y = next.fetch_add(1);
                if (y >= fp.row_end) break;
                for (int x = 0; x < fp.width; x++) {
                    st.add(rm::C_PIXELS);
                    int pid;
                    const rm::Vec3<R> dir = vw.apply(rm::backproject<R>(fp, x, y));
                    const rm::Vec3<R> c = rm::cast_ray<R, true, rm::SceneView<R>>(sc, fp.camera, dir, fp.background, fp.max_depth, pid, st);
                    const size_t px = (size_t)y * fp.width + x;
                    out_rgb[3 * px] = c.x; out_rgb[3 * px + 1] = c.y; out_rgb[3 * px + 2] = c.z;
                    if (prim) prim[px] = pid;
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        uint64_t* dst = &stats->pixels;
        for (auto& c : tc) for (int i = 0; i < rm::C_COUNT; i++) dst[i] += c.c[i];
    }
    return RM_OK;
}

}  // namespace

extern "C" {
// basis: u, v, w as rm_view_basis writes them
int emu_render_fast_view(const RmFlatScene* fs, const RmParams* p, const double basis[9], float* out_rgb, int32_t* prim, int n_threads) {
    const rm::ViewBasis vw = view_basis_of(basis);
    return p->accel && fs->n_lights <= rm::kBvhMaxLights ? emu_render_fast_view_impl<true>(fs, p, vw, out_rgb, prim, n_threads)
                                                         : emu_render_fast_view_impl<false>(fs, p, vw, out_rgb, prim, n_threads);
}
int emu_render_f64_view(const RmFlatScene* fs, const RmParams* p, const double basis[9], double* out_rgb, int32_t* prim, RmStats* stats,
                        int n_threads) {
    return emu_render_view_impl<double>(fs, p, view_basis_of(basis), out_rgb, prim, stats, n_threads);
}
int emu_view_basis(const RmView* view, double out[9]) {
    const char* err = "";
    return rm::view_basis(*view, out, &err);
}
}
