// rm_distributed.cu -- the distributed ray tracing kernel (rm_render_distributed, include/rm_b200.h) and its launcher: lens,
// area lights, rough glass and motion in one frame, sampled_kernel (rm_sampled.cuh) with distributed_kernel::Effect.  A
// translation unit of its own, like rm_lens.cu: instantiated next to other kernels it would change how the compiler optimises
// their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Distributed ray tracing (rm_render_distributed) ---------------------------------------------------------------------
// Every query, surface and shadow ray on DistributedView for sample q = i s + j: at the sample's time tau = mo.tau[q] when
// kMotion (MotionView, the swept hierarchy), in the uploaded scene otherwise, and with the area lights' point of
// area_offset(s, i, j, L) at every level L.  The recursion is cast_glass_distributed, rough glass's turn included (rg.g null:
// nothing is rough).  The hit queue holds the ray index, which gives q again when the hit is shaded.
namespace distributed_kernel {
template <bool kMotion> struct Effect {
    static constexpr int kNoneSlot = GLASS_NONE;
    AreaPoints ap;
    RoughGlass rg;
    Motion mo;
    template <bool kBvh>
    static __device__ __forceinline__ bool query(const FastViewT<kBvh, false>& fv, const Effect& eff, const int s,
                                                 const int r, const Vec3<double>& o, const Vec3<double>& d, HitRec<float>& h,
                                                 Counters<false>& st) {
        const DistributedView<kBvh, kMotion> dv(fv, eff.mo, eff.ap, r % (s * s));
        return dv.template closest<false>(to_f32(o), to_f32(d), 1, h, st);
    }
    template <int kGlass, bool kBvh>
    static __device__ __forceinline__ Vec3<float> shade(const FastViewT<kBvh, false>& fv, const FrameParams<float>& fp,
                                                        const Effect& eff, const int s, const int r, const Vec3<double>& o,
                                                        const Vec3<double>& d, const HitRec<float>& h) {
        const DistributedView<kBvh, kMotion> dv(fv, eff.mo, eff.ap, r % (s * s));
        return distributed_shade<kGlass>(dv, fp, eff.rg, o, d, h);
    }
};

}  // namespace distributed_kernel

}  // namespace

cudaError_t launch_distributed(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const AreaPoints& ap,
                               const RoughGlass& rg, const Motion& mo, const bool motion, const double reach, bool cull, long long n_px,
                               unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream) {
    if (!motion) return launch_sampled(ds, fp, lc, distributed_kernel::Effect<false>{ap, rg, mo}, reach, cull, n_px, next, rgb, dmax, stream);
    return launch_sampled(ds, fp, lc, distributed_kernel::Effect<true>{ap, rg, mo}, reach, cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
