// rm_motion.cu -- the motion-blur kernel (rm_render_motion, include/rm_b200.h RmMotion) and its launcher: sampled_kernel
// (rm_sampled.cuh) with motion_kernel::Effect.  A translation unit of its own, like rm_lens.cu: instantiated next to other
// kernels it would change how the compiler optimises their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Motion blur (rm_render_motion) ---------------------------------------------------------------------------------------
// Every query at the sample's own time: each sample ray -- its level-1 query, the recursion and every shadow ray -- runs on
// MotionView at tau = mo.tau[q] of its sample q = i s + j, through lens_shade unchanged.  The hit queue holds the ray index,
// which gives q, and with it tau, again when the hit is shaded.
namespace motion_kernel {
struct Effect {
    static constexpr int kNoneSlot = GLASS_NONE;
    Motion mo;
    template <bool kBvh>
    static __device__ __forceinline__ bool query(const FastViewT<kBvh, false>& fv, const Effect& eff, const int s, const int r,
                                                 const Vec3<double>& o, const Vec3<double>& d, HitRec<float>& h, Counters<false>& st) {
        const MotionView<kBvh> mv(fv, eff.mo, r % (s * s));
        return mv.template closest<false>(to_f32(o), to_f32(d), 1, h, st);
    }
    template <int kGlass, bool kBvh>
    static __device__ __forceinline__ Vec3<float> shade(const FastViewT<kBvh, false>& fv, const FrameParams<float>& fp,
                                                        const Effect& eff, const int s, const int r, const Vec3<double>& o,
                                                        const Vec3<double>& d, const HitRec<float>& h) {
        const MotionView<kBvh> mv(fv, eff.mo, r % (s * s));
        return lens_shade<kGlass>(mv, fp, o, d, h);
    }
};

}  // namespace motion_kernel

}  // namespace

cudaError_t launch_motion(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const Motion& mo,
                          const double reach, bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax,
                          cudaStream_t stream) {
    return launch_sampled(ds, fp, lc, motion_kernel::Effect{mo}, reach, cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
