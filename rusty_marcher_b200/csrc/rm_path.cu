// rm_path.cu -- the path-traced kernel (rm_render_path, include/rm_b200.h) and its launcher: diffuse interreflection with
// lens, area lights, rough glass and motion in one frame, sampled_kernel (rm_sampled.cuh) with path_kernel::Effect.  A
// translation unit of its own, like rm_lens.cu: instantiated next to other kernels it would change how the compiler optimises
// their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Path-traced frames (rm_render_path) ---------------------------------------------------------------------------------
// distributed_kernel::Effect's queries with cast_path as the recursion: every query, surface and shadow ray on DistributedView for
// sample q = i s + j (at the sample's time tau = mo.tau[q] when kMotion, through the swept hierarchy; the area lights' point
// of area_offset(s, i, j, L) at every level L), rough glass's turn (rg.g null: nothing is rough) and one diffuse bounce per
// qualifying opaque hit at the disc points df.  Opaque hits recurse here, so all three glass modes exist: GLASS_NONE traces
// the bounces in FP32 without the glass branch.
namespace path_kernel {
template <bool kMotion> struct Effect {
    static constexpr int kNoneSlot = GLASS_NONE;
    AreaPoints ap;
    RoughGlass rg;
    Motion mo;
    Diffuse df;
    template <bool kBvh>
    static __device__ __forceinline__ bool query(const FastViewT<kBvh, false>& fv, const Effect& eff, const int s, const int r,
                                                 const Vec3<double>& o, const Vec3<double>& d, HitRec<float>& h, Counters<false>& st) {
        const DistributedView<kBvh, kMotion> dv(fv, eff.mo, eff.ap, r % (s * s));
        return dv.template closest<false>(to_f32(o), to_f32(d), 1, h, st);
    }
    template <int kGlass, bool kBvh>
    static __device__ __forceinline__ Vec3<float> shade(const FastViewT<kBvh, false>& fv, const FrameParams<float>& fp,
                                                        const Effect& eff, const int s, const int r, const Vec3<double>& o,
                                                        const Vec3<double>& d, const HitRec<float>& h) {
        const DistributedView<kBvh, kMotion> dv(fv, eff.mo, eff.ap, r % (s * s));
        return path_shade<kGlass>(dv, fp, eff.rg, eff.df, o, d, h);
    }
};

}  // namespace path_kernel

}  // namespace

cudaError_t launch_path(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const AreaPoints& ap,
                        const RoughGlass& rg, const Motion& mo, const Diffuse& df, const bool motion, const double reach, bool cull,
                        long long n_px, unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream) {
    if (!motion) return launch_sampled(ds, fp, lc, path_kernel::Effect<false>{ap, rg, mo, df}, reach, cull, n_px, next, rgb, dmax, stream);
    return launch_sampled(ds, fp, lc, path_kernel::Effect<true>{ap, rg, mo, df}, reach, cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
