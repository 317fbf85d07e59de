// rm_indirect_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// The diffuse interreflection of rm_render_indirect through the product's own code compiled for the host, next to rm_emu.cpp
// (included here unchanged): make_lens_camera and rm::lens_ray build each sample ray in f64, FastViewT::closest (brute force or
// the hierarchy) finds its level-1 hit in FP32, indirect_shade traces the recursion with its bounces in the glass mode the
// launcher picks (GLASS_NONE included), and rm::resolve_box averages the samples -- the per-ray device code of indirect_kernel.
// Nothing is routed: every call runs the indirect code, whatever the scene and max_depth.
#include "rm_emu.cpp"

namespace {

template <int S> void resolve_pixel(const float* v, float out[3]) {
    rm::resolve_box<S>([&](int i, float (&row)[3 * S]) {
        for (int c = 0; c < 3 * S; c++) row[c] = v[3 * i * S + c];
    }, out);
}

template <bool kBvh>
int emu_render_indirect_impl(const RmFlatScene* fs, const RmParams* p, const double* basis, const RmLens& lens, float* out_rgb,
                             int n_threads) {
    rm::PackedScene<float> ps;
    std::string err;
    int rc = rm::pack_scene<float>(*fs, ps, err);
    if (rc != RM_OK) return rc;
    if (p->width % 32) return RM_ERR_DIMENSIONS;
    const bool cull = p->cull_backfacing != 0;
    const rm::BlobLayout& L = ps.lay;
    const unsigned char* base = ps.blob_data();
    rm::FastViewT<kBvh> fv0;
    fv0.bvh.nodes = ps.bvh_nodes.data();
    fv0.bvh.prims = ps.bvh_prims.data();
    fv0.bvh.n_nodes = (int)(ps.bvh_nodes.size() / 4);
    fv0.sph = reinterpret_cast<const rm::R4<float>*>(base + L.off_sph);
    fv0.sph_id = reinterpret_cast<const int*>(base + L.off_sph_id);
    fv0.n_sph = L.n_sph;
    fv0.tri_g = reinterpret_cast<const rm::R4<float>*>(base + L.off_tri_g);
    fv0.tri_r = nullptr;                                        // (the sample rays do not start at the camera)
    fv0.n_tri = rm::tri_count(L, cull);
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
    const rm::LensCamera lc = rm::make_lens_camera(*p, basis, lens);
    const rm::Diffuse df = rm::make_diffuse(lens.samples);
    const double extent[3] = {fabs(lc.cam[0]) + lc.aperture, fabs(lc.cam[1]) + lc.aperture, fabs(lc.cam[2]) + lc.aperture};
    const int gm = g_glass_mode.load() >= 0 ? g_glass_mode.load() : rm::glass_mode(L.any_glass != 0, L.n_sph, L.coord_max, L.r_min, extent);
    g_last_glass_mode.store(gm);
    const int s = lens.samples, ss = s * s;
    std::atomic<int> next{fp.row_begin};
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; t++) {
        pool.emplace_back([&] {
            rm::FastViewT<kBvh> fv = fv0;
            std::vector<float> v(3 * ss);
            for (;;) {
                const int y = next.fetch_add(1);
                if (y >= fp.row_end) break;
                for (int x = 0; x < fp.width; x++) {
                    for (int q = 0; q < ss; q++) {
                        rm::Vec3<double> o, d;
                        rm::lens_ray(lc, x, y, q / s, q % s, o, d);
                        rm::HitRec<float> h;
                        rm::Counters<false> st;
                        rm::Vec3<float> c = {0.f, 0.f, 0.f};
                        if (fv.template closest<false>(rm::to_f32(o), rm::to_f32(d), 1, h, st))
                            c = gm == rm::GLASS_NONE  ? rm::indirect_shade<rm::GLASS_NONE>(fv, fp, df, q / s, q % s, o, d, h)
                                : gm == rm::GLASS_F32 ? rm::indirect_shade<rm::GLASS_F32>(fv, fp, df, q / s, q % s, o, d, h)
                                                      : rm::indirect_shade<rm::GLASS_F64>(fv, fp, df, q / s, q % s, o, d, h);
                        v[3 * q] = c.x; v[3 * q + 1] = c.y; v[3 * q + 2] = c.z;
                    }
                    float* dst = out_rgb + 3 * ((size_t)y * fp.width + x);
                    switch (s) {
                        case 1: resolve_pixel<1>(v.data(), dst); break;
                        case 2: resolve_pixel<2>(v.data(), dst); break;
                        case 3: resolve_pixel<3>(v.data(), dst); break;
                        case 4: resolve_pixel<4>(v.data(), dst); break;
                        case 5: resolve_pixel<5>(v.data(), dst); break;
                        case 6: resolve_pixel<6>(v.data(), dst); break;
                        case 7: resolve_pixel<7>(v.data(), dst); break;
                        default: resolve_pixel<8>(v.data(), dst); break;
                    }
                }
            }
        });
    }
    for (auto& th : pool) th.join();
    return RM_OK;
}

}  // namespace

extern "C" {
void emu_diffuse_offset(int s, int i, int j, int level, double out[2]) { rm::diffuse_offset(s, i, j, level, &out[0], &out[1]); }

// the bounce direction and origin at a hit (point, hit normal) of a ray of direction d, with the disc point (lx, ly)
void emu_diffuse_ray(const double point[3], const double hit_normal[3], const double d[3], double lx, double ly, double o_out[3],
                     double d_out[3]) {
    const rm::Vec3<double> p = {point[0], point[1], point[2]}, n = {hit_normal[0], hit_normal[1], hit_normal[2]};
    const rm::Vec3<double> nf = rm::diffuse_normal<double>(n, {d[0], d[1], d[2]});
    const rm::Vec3<double> o = rm::diffuse_origin<double>(p, nf), r = rm::diffuse_dir<double>(nf, lx, ly);
    o_out[0] = o.x; o_out[1] = o.y; o_out[2] = o.z;
    d_out[0] = r.x; d_out[1] = r.y; d_out[2] = r.z;
}

// the FP32 indirect frame over the patch rows of p (rows outside untouched); basis: u, v, w, or null
int emu_render_indirect(const RmFlatScene* fs, const RmParams* p, const double* basis, const RmLens* lens, float* out_rgb,
                        int n_threads) {
    return p->accel && fs->n_lights <= rm::kBvhMaxLights ? emu_render_indirect_impl<true>(fs, p, basis, *lens, out_rgb, n_threads)
                                                         : emu_render_indirect_impl<false>(fs, p, basis, *lens, out_rgb, n_threads);
}
}
