// rm_area_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// The spherical area lights of rm_render_area_lights through the product's own code compiled for the host, next to rm_emu.cpp
// (included here unchanged): prepare_raster and stage A one pixel at a time (primary_begin, primary_tri, primary_rest, or
// primary_bvh), then fast_shade on rm::AreaView in the glass mode the launcher picks -- the per-pixel device code of
// area_light_kernel, with the AreaLights the library builds.
#include <cfloat>

#include "rm_emu.cpp"

namespace {

rm::AreaLights area_lights(const double* radius, int n, int s, std::vector<float>& r32) {
    rm::AreaLights al = {};
    r32.assign(std::max(n, 1), 0.f);
    for (int l = 0; l < n; l++) r32[l] = radius[l] > 0. ? std::max((float)std::min(radius[l], (double)FLT_MAX), 1e-30f) : 0.f;
    for (int a = 0; a < s; a++)
        for (int b = 0; b < s; b++) {
            double lx, ly;
            rm::lens_offset(s, a, b, &lx, &ly);
            al.off[2 * (a * s + b)] = (float)lx;
            al.off[2 * (a * s + b) + 1] = (float)ly;
        }
    al.radius = r32.data();
    al.samples = s;
    al.inv_ss = 1.f / (float)(s * s);
    return al;
}

template <bool kBvh>
int emu_render_area_impl(const RmFlatScene* fs, const RmParams* p, const double* radius, int s, float* out_rgb, int32_t* prim, int n_threads) {
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
    for (int j = 0; j < n_tri; j++) rm::prepare_raster(ps.tri_src.data() + (size_t)j * rm::kTriSrcDoubles, p->camera, tri_r.data() + 4 * j);
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
    std::vector<float> r32;
    const rm::AreaLights al = area_lights(radius, L.n_lgt, s, r32);
    const rm::FrameParams<float> fp = rm::make_frame_params<float>(*p);
    const int gm = g_glass_mode.load() >= 0 ? g_glass_mode.load() : rm::glass_mode(L.any_glass != 0, L.n_sph, L.coord_max, L.r_min, p->camera);
    g_last_glass_mode.store(gm);
    std::atomic<int> next{fp.row_begin};
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) {
        pool.emplace_back([&] {
            rm::FastViewT<kBvh> fv = fv0;
            const rm::AreaView<rm::FastViewT<kBvh>> av(fv, al);
            for (;;) {
                const int y = next.fetch_add(1);
                if (y >= fp.row_end) break;
                for (int x = 0; x < fp.width; x++) {
                    rm::PrimaryState<1> st;
                    rm::primary_begin<1>(st, fp, x, y);
                    if constexpr (kBvh) {
                        rm::primary_bvh<1>(st, fv, fp);
                    } else {
                        for (int j = 0; j < n_tri; j++) rm::primary_tri<1>(st, tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], fv.n_sph + j);
                        if (fv.n_sph + fv.n_poly > 0) rm::primary_rest<1>(st, fv, fp);
                    }
                    rm::Vec3<float> c = {0.f, 0.f, 0.f};
                    if (st.slot[0] >= 0)
                        c = gm == rm::GLASS_NONE  ? rm::fast_shade<rm::GLASS_NONE>(av, fp, x, y, st.t[0], st.slot[0], st.id[0])
                            : gm == rm::GLASS_F32 ? rm::fast_shade<rm::GLASS_F32>(av, fp, x, y, st.t[0], st.slot[0], st.id[0])
                                                  : rm::fast_shade<rm::GLASS_F64>(av, fp, x, y, st.t[0], st.slot[0], st.id[0]);
                    const size_t px = (size_t)y * fp.width + x;
                    out_rgb[3 * px] = c.x; out_rgb[3 * px + 1] = c.y; out_rgb[3 * px + 2] = c.z;
                    if (prim) prim[px] = st.id[0];
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    return RM_OK;
}

}  // namespace

extern "C" {
// the normative f64 definition (rm::light_frame<double> / rm::light_sample<double>) as the library compiles it
void emu_light_frame(const double m[3], double t1[3], double t2[3]) {
    rm::Vec3<double> a, b;
    rm::light_frame<double>(rm::Vec3<double>{m[0], m[1], m[2]}, a, b);
    t1[0] = a.x; t1[1] = a.y; t1[2] = a.z;
    t2[0] = b.x; t2[1] = b.y; t2[2] = b.z;
}
void emu_light_sample(const double c[3], double r, const double t1[3], const double t2[3], double lx, double ly, double q[3]) {
    const rm::Vec3<double> v = rm::light_sample<double>(rm::Vec3<double>{c[0], c[1], c[2]}, r, rm::Vec3<double>{t1[0], t1[1], t1[2]},
                                                        rm::Vec3<double>{t2[0], t2[1], t2[2]}, lx, ly);
    q[0] = v.x; q[1] = v.y; q[2] = v.z;
}

// the FP32 area-light frame over the patch rows of p (rows outside untouched); radius: one per light
int emu_render_area(const RmFlatScene* fs, const RmParams* p, const double* radius, int samples, float* out_rgb, int32_t* prim, int n_threads) {
    return p->accel && fs->n_lights <= rm::kBvhMaxLights ? emu_render_area_impl<true>(fs, p, radius, samples, out_rgb, prim, n_threads)
                                                         : emu_render_area_impl<false>(fs, p, radius, samples, out_rgb, prim, n_threads);
}
}
