// rm_path_emu.cpp -- DEV/TEST TOOL, not part of the product and never loaded by it.
//
// The path-traced frame of rm_render_path through the product's own code compiled for the host, next to rm_emu.cpp (included
// here unchanged): make_area_points, make_rough_glass, make_diffuse, rm::motion_displacements and rm::make_motion lay out the
// effects and the bounce's disc points as the kernel reads them, rm::build_swept_bvh builds the swept hierarchy,
// make_lens_camera and rm::lens_ray build each sample ray in f64, rm::DistributedView for the sample answers its level-1 query
// and, through path_shade, the recursion with its bounces and the shadow rays in the glass mode the launcher picks (GLASS_NONE
// included), and rm::resolve_box averages the samples -- the per-ray device code of path_kernel.  Nothing is routed: every
// call runs the path code, whatever the scene, the effects and max_depth.
#include "rm_emu.cpp"

namespace {

template <int S> void resolve_pixel(const float* v, float out[3]) {
    rm::resolve_box<S>([&](int i, float (&row)[3 * S]) {
        for (int c = 0; c < 3 * S; c++) row[c] = v[3 * i * S + c];
    }, out);
}

template <bool kBvh, bool kMotion>
int emu_render_path_impl(const RmFlatScene* fs, const RmParams* p, const double* basis, const RmLens& lens, const double* radius,
                         const double* roughness, int n_rough, const double* disp, float* out_rgb, int n_threads) {
    rm::PackedScene<float> ps;
    std::string err;
    int rc = rm::pack_scene<float>(*fs, ps, err);
    if (rc != RM_OK) return rc;
    if (p->width % 32) return RM_ERR_DIMENSIONS;
    const bool cull = p->cull_backfacing != 0;
    const rm::BlobLayout& L = ps.lay;
    const unsigned char* base = ps.blob_data();
    std::vector<rm::R4<float>> vel;
    double reach = 0.;
    std::vector<rm::R4<float>> nodes = ps.bvh_nodes;
    std::vector<int> prims = ps.bvh_prims;
    if (kMotion) {
        rm::motion_displacements(ps, disp, vel, reach);
        if (kBvh) rm::build_swept_bvh(ps, vel, nodes, prims);
    }
    rm::FastViewT<kBvh> fv0;
    fv0.bvh.nodes = nodes.data();
    fv0.bvh.prims = prims.data();
    fv0.bvh.n_nodes = (int)(nodes.size() / 4);
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
    const int s = lens.samples, ss = s * s;
    std::vector<float> r32, g32;
    rm::AreaPoints ap = rm::make_area_points(s, radius, radius ? fs->n_lights : 0, r32);
    r32.resize(std::max<size_t>(r32.size(), (size_t)fs->n_lights), 0.f);
    ap.radius = r32.data();
    rm::RoughGlass rg = rm::make_rough_glass(s, roughness, roughness ? n_rough : 0, g32);
    rg.g = roughness ? g32.data() : nullptr;
    const rm::Diffuse df = rm::make_diffuse(s);
    rm::Motion mo = rm::make_motion(s);
    if (kMotion) {
        mo.v_sph = vel.data();
        mo.v_tri = vel.data() + L.n_sph;
        mo.v_pln = vel.data() + L.n_sph + L.n_tri;
    }
    // (the launcher's plan: the camera's extent widened by the aperture, the scene's coordinates by the reach of the motion)
    const double extent[3] = {fabs(lc.cam[0]) + lc.aperture, fabs(lc.cam[1]) + lc.aperture, fabs(lc.cam[2]) + lc.aperture};
    const int gm = g_glass_mode.load() >= 0 ? g_glass_mode.load()
                                            : rm::glass_mode(L.any_glass != 0, L.n_sph, L.coord_max + reach, L.r_min, extent);
    g_last_glass_mode.store(gm);
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
                        const rm::DistributedView<kBvh, kMotion> dv(fv, mo, ap, q);
                        rm::HitRec<float> h;
                        rm::Counters<false> st;
                        rm::Vec3<float> c = {0.f, 0.f, 0.f};
                        if (dv.template closest<false>(rm::to_f32(o), rm::to_f32(d), 1, h, st))
                            c = gm == rm::GLASS_NONE  ? rm::path_shade<rm::GLASS_NONE>(dv, fp, rg, df, o, d, h)
                                : gm == rm::GLASS_F32 ? rm::path_shade<rm::GLASS_F32>(dv, fp, rg, df, o, d, h)
                                                      : rm::path_shade<rm::GLASS_F64>(dv, fp, rg, df, o, d, h);
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
// the FP32 path-traced frame over the patch rows of p (rows outside untouched); basis: u, v, w, or null; radius: one per light
// of the scene, roughness: n_rough values by primitive id, disp: 3 values per primitive id -- each null for no such effect.
// disp given runs the motion code (MotionView, the swept hierarchy), whatever its values.
int emu_render_path(const RmFlatScene* fs, const RmParams* p, const double* basis, const RmLens* lens, const double* radius,
                    const double* roughness, int n_rough, const double* disp, float* out_rgb, int n_threads) {
    const bool bvh = p->accel && fs->n_lights <= rm::kBvhMaxLights;
    if (disp) return bvh ? emu_render_path_impl<true, true>(fs, p, basis, *lens, radius, roughness, n_rough, disp, out_rgb, n_threads)
                         : emu_render_path_impl<false, true>(fs, p, basis, *lens, radius, roughness, n_rough, disp, out_rgb, n_threads);
    return bvh ? emu_render_path_impl<true, false>(fs, p, basis, *lens, radius, roughness, n_rough, disp, out_rgb, n_threads)
               : emu_render_path_impl<false, false>(fs, p, basis, *lens, radius, roughness, n_rough, disp, out_rgb, n_threads);
}
}
