// rm_indirect.cu -- the diffuse interreflection kernel (rm_render_indirect, include/rm_b200.h) and its launcher: sampled_kernel
// (rm_sampled.cuh) with indirect_kernel::Effect.  A translation unit of its own, like rm_lens.cu: instantiated next to other
// kernels it would change how the compiler optimises their shared inline code, and with it their machine code.
#include "rm_sampled.cuh"

namespace rm {

namespace {

// ---- Diffuse interreflection (rm_render_indirect) -------------------------------------------------------------------------
// The thin-lens camera's queries (FastViewT::closest), shaded by indirect_shade: cast_indirect as the recursion, one diffuse
// bounce per qualifying opaque hit at the disc points df of sample (i, j).  Opaque hits recurse here, so all three glass modes
// exist: GLASS_NONE traces the bounces in FP32 without the glass branch.
namespace indirect_kernel {
struct Effect {
    static constexpr int kNoneSlot = GLASS_NONE;
    Diffuse df;
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
        return indirect_shade<kGlass>(fv, fp, eff.df, q / s, q % s, o, d, h);
    }
};

}  // namespace indirect_kernel

}  // namespace

cudaError_t launch_indirect(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const Diffuse& df,
                            bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream) {
    return launch_sampled(ds, fp, lc, indirect_kernel::Effect{df}, 0., cull, n_px, next, rgb, dmax, stream);
}

}  // namespace rm
