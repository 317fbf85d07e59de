// rm_rough.cu -- the rough-glass kernel (rm_render_rough_glass, include/rm_b200.h RmRoughGlass) and its launcher:
// sampled_kernel (rm_sampled.cuh) with rough_glass_kernel::Effect.  A translation unit of its own, like rm_lens.cu: instantiated
// next to other kernels it would change how the compiler optimises their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Rough glass (rm_render_rough_glass) ----------------------------------------------------------------------------------
// The thin-lens camera's queries (FastViewT::closest), shaded by rough_shade: cast_glass_rough as the recursion, its turns by
// the roughness rg at sample (i, j).
namespace rough_glass_kernel {
struct Effect {
    // only scenes with a rough glass-like primitive come here, so the glass mode is GLASS_F32 or GLASS_F64; the GLASS_NONE slot
    // holds the FP32 recursion (an opaque hit leaves it after its direct lighting)
    static constexpr int kNoneSlot = GLASS_F32;
    RoughGlass rg;
    template <bool kBvh>
    static __device__ __forceinline__ bool query(const FastViewT<kBvh, false>& fv, const Effect&, const int, const int,
                                                 const Vec3<double>& o, const Vec3<double>& d, HitRec<float>& h, Counters<false>& st) {
        return fv.template closest<false>(to_f32(o), to_f32(d), 1, h, st);
    }
    template <int kGlass, bool kBvh>
    static __device__ __forceinline__ Vec3<float> shade(const FastViewT<kBvh, false>& fv, const FrameParams<float>& fp,
                                                        const Effect& eff, const int s, const int r, const Vec3<double>& o,
                                                        const Vec3<double>& d, const HitRec<float>& h) {
        const int q = r % (s * s);
        return rough_shade<kGlass>(fv, fp, eff.rg, q / s, q % s, o, d, h);
    }
};

}  // namespace rough_glass_kernel

}  // namespace

cudaError_t launch_rough_glass(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const RoughGlass& rg,
                               bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream) {
    return launch_sampled(ds, fp, lc, rough_glass_kernel::Effect{rg}, 0., cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
