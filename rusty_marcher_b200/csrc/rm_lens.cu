// rm_lens.cu -- the thin-lens camera's kernel (rm_render_lens, include/rm_b200.h RmLens) and its launcher: sampled_kernel
// (rm_sampled.cuh) with lens_kernel::Effect.  A translation unit of its own: instantiated next to K1 and the adaptive sub-pixel
// kernel it changes how the compiler optimises their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Thin-lens camera (rm_render_lens) ------------------------------------------------------------------------------------
// Every query on the general closest-hit query (FastViewT::closest, brute force or the hierarchy), shaded by lens_shade.
namespace lens_kernel {
struct Effect {
    static constexpr int kNoneSlot = GLASS_NONE;
    template <bool kBvh>
    static __device__ __forceinline__ bool query(const FastViewT<kBvh, false>& fv, const Effect&, const int, const int,
                                                 const Vec3<double>& o, const Vec3<double>& d, HitRec<float>& h, Counters<false>& st) {
        return fv.template closest<false>(to_f32(o), to_f32(d), 1, h, st);
    }
    template <int kGlass, bool kBvh>
    static __device__ __forceinline__ Vec3<float> shade(const FastViewT<kBvh, false>& fv, const FrameParams<float>& fp, const Effect&,
                                                        const int, const int, const Vec3<double>& o, const Vec3<double>& d,
                                                        const HitRec<float>& h) {
        return lens_shade<kGlass>(fv, fp, o, d, h);
    }
};

}  // namespace lens_kernel

}  // namespace

cudaError_t launch_lens(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, bool cull, long long n_px,
                        unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream) {
    return launch_sampled(ds, fp, lc, lens_kernel::Effect{}, 0., cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
