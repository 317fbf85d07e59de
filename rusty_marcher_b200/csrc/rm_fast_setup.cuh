// rm_fast_setup.cuh -- what the kernels over FastViewT share (rm_kernels.cu: K1 and the adaptive sub-pixel kernel; rm_sampled.cuh:
// the sampled-frame kernel): the CTA shape, the staging of the scene in shared memory and the view of it, and on the host
// the launch plan and the one-time set-up of a kernel family.
#pragma once

#include <algorithm>
#include <cassert>
#include <initializer_list>

#include "rm_kernels.h"

// -DRM_CHECKED: bounds and protocol checks inside the kernels (device assert: file, line, block and thread on stderr, then
// the kernel traps and the next CUDA call fails).  compute-sanitizer is closed on this project's GPU pool, so this is the
// memory-safety pass that can be run there: tools/gpu_checked.sh builds the variant and runs the GPU suite with it.
#ifdef RM_CHECKED
#define RM_CHECK(cond) assert(cond)
#else
#define RM_CHECK(cond) ((void)0)
#endif

namespace rm {

namespace {

constexpr int kSmemLimit = 200 * 1024;

__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));            // v >= 0: int order == float order
}
__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v) {
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// CTA shape of the render kernel.  The shading stage wants ~116 registers to run without spills, and it is bound by
// instruction latency and spill traffic rather than by the number of resident warps: measured on the cornell / demo /
// dodecahedron frames (render phase, us) -- 3 CTAs x 8 warps at 80 registers 55 / 205 / 49, 5 x 4 warps at 96 registers
// 54 / 194 / 44, 2 x 8 warps at 128 registers 53 / 174 / 40 (gpurun_out/ab_r2a.log).  Hence two CTAs of eight warps.
#ifndef RM_K1_BLOCK
#define RM_K1_BLOCK 256
#endif
#ifndef RM_K1_MIN_BLOCKS
#define RM_K1_MIN_BLOCKS 2                                      // resident CTAs per SM the register allocation aims at
#endif
constexpr int kFastBlock = RM_K1_BLOCK;

// The scene in shared memory of K1, adaptive_subpixel_kernel and sampled_kernel (kSmem): blob | raster records of every
// fast-path triangle | materials mat_a | mat_b | mat_f (stage_mat: if they fit as well).  The kernels stage and view it with
// these helpers, so that a sub-pixel value of the adaptive kernel stays the value K1 writes for that pixel.
// The static part, blob and materials, does not depend on K0 (sampled_kernel stages only this part).
__device__ __forceinline__ void stage_static(const DeviceScene<float>& ds, const int stage_mat, unsigned char* smem_raw) {
    const BlobLayout& L = ds.lay;
    const uint4* src = reinterpret_cast<const uint4*>(ds.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem_raw);
    const int n16 = L.bytes / 16;
    for (int i = threadIdx.x; i < n16; i += kFastBlock) dst[i] = __ldg(src + i);
    if (stage_mat) {                                            // materials behind the raster records: mat_a | mat_b | mat_f
        uint4* m = dst + n16 + L.n_tri * 4;
        const uint4* a = reinterpret_cast<const uint4*>(ds.mat_a);
        const uint4* b = reinterpret_cast<const uint4*>(ds.mat_b);
        for (int i = threadIdx.x; i < ds.n_mat; i += kFastBlock) {
            m[i] = __ldg(a + i);
            m[ds.n_mat + i] = __ldg(b + i);
            reinterpret_cast<int*>(m + 2 * ds.n_mat)[i] = __ldg(ds.mat_f + i);
        }
    }
}
// The raster records K0 wrote; base and tri_r then point into shared memory.
__device__ __forceinline__ void stage_raster(const DeviceScene<float>& ds, const int n_tri, unsigned char* smem_raw,
                                             const unsigned char*& base, const R4<float>*& tri_r) {
    uint4* dst = reinterpret_cast<uint4*>(smem_raw);
    const int n16 = ds.lay.bytes / 16;
    const uint4* rsrc = reinterpret_cast<const uint4*>(ds.tri_r);
    for (int i = threadIdx.x; i < n_tri * 4; i += kFastBlock) dst[n16 + i] = rsrc[i];
    base = smem_raw;
    tri_r = reinterpret_cast<const R4<float>*>(smem_raw + ds.lay.bytes);
}
// The scene as the fast device functions read it: the blob's arrays from base (ds.blob or its staged copy), the n_tri
// raster records from tri_r, the materials from shared memory if they were staged (smem_mat).  n_tri is the caller's
// tri_count(): computed again here, it changes K1's machine code.
template <bool kBvh, bool kCount>
__device__ __forceinline__ FastViewT<kBvh, kCount> make_fast_view(const DeviceScene<float>& ds, const unsigned char* base,
                                                                  const R4<float>* tri_r, const int n_tri, const int cull,
                                                                  const bool smem_mat, const unsigned char* smem_raw) {
    const BlobLayout& L = ds.lay;
    FastViewT<kBvh, kCount> fv;
    fv.bvh = ds.bvh;
    fv.sph = reinterpret_cast<const R4<float>*>(base + L.off_sph);
    fv.sph_id = reinterpret_cast<const int*>(base + L.off_sph_id);
    fv.n_sph = L.n_sph;
    fv.tri_g = reinterpret_cast<const R4<float>*>(base + L.off_tri_g);
    fv.tri_r = tri_r;
    fv.n_tri = n_tri;
    fv.poly_slot = reinterpret_cast<const int*>(base + L.off_poly_slot);
    fv.n_poly = poly_count(L, cull != 0);
    fv.pln_n = reinterpret_cast<const R4<float>*>(base + L.off_pln_n);
    fv.pln_c = reinterpret_cast<const R4<float>*>(base + L.off_pln_c);
    fv.pln_v = reinterpret_cast<const I2*>(base + L.off_pln_v);
    fv.pln_id = reinterpret_cast<const int*>(base + L.off_pln_id);
    fv.vert = reinterpret_cast<const R4<float>*>(base + L.off_vert);
    fv.mat_a = ds.mat_a;
    fv.mat_b = ds.mat_b;
    fv.mat_f = ds.mat_f;
    if (smem_mat) {
        fv.mat_a = reinterpret_cast<const R4<float>*>(smem_raw + L.bytes + (size_t)L.n_tri * 64);
        fv.mat_b = fv.mat_a + ds.n_mat;
        fv.mat_f = reinterpret_cast<const int*>(fv.mat_b + ds.n_mat);
    }
    fv.lgt_p = reinterpret_cast<const R4<float>*>(base + L.off_lgt_p);
    fv.lgt_c = reinterpret_cast<const R4<float>*>(base + L.off_lgt_c);
    fv.n_lgt = L.n_lgt;
    fv.sph64 = ds.sph64;
    fv.tri64 = ds.tri_src;
    fv.pln64 = ds.pln64;
    return fv;
}

// The launch plan of K1, adaptive_subpixel_kernel and sampled_kernel: it picks the instantiation, and a sub-pixel value of the
// adaptive kernel is the value K1 writes for that pixel only while both kernels pick alike.
// Shared memory: scene blob | raster records of every fast-path triangle | materials (if they fit as well), next to the
// kernel's static arrays (hit queues etc.) within dyn_limit.
struct FastPlan {
    bool bvh;                                                   // walk the hierarchy
    bool use_smem;                                              // stage the scene in shared memory
    int stage_mat;                                              // ... the materials as well
    int glass;                                                  // GlassMode
    size_t dyn_smem;                                            // dynamic shared memory of the launch
    int row() const { return bvh ? 2 : use_smem ? 0 : 1; }      // of the instantiation tables: staged | global | hierarchy
};

FastPlan fast_plan(const DeviceScene<float>& ds, const FrameParams<float>& fp, const double camera[3], const int dyn_limit) {
    FastPlan p;
    p.bvh = fp.accel != 0 && ds.bvh.n_nodes > 0 && ds.lay.n_lgt <= kBvhMaxLights;
    const size_t smem_geo = (size_t)ds.lay.bytes + (size_t)ds.lay.n_tri * 64;
    const size_t smem_mat = (((size_t)ds.n_mat * 36) + 15) / 16 * 16;
    p.stage_mat = smem_geo + smem_mat <= (size_t)dyn_limit ? 1 : 0;
    const size_t smem = smem_geo + (p.stage_mat ? smem_mat : 0);
    p.use_smem = !p.bvh && smem <= (size_t)dyn_limit;
    // the reflect / refract recursion only where a frame can need it, its f64 ray geometry only where FP32 would not do
    p.glass = glass_mode(ds.lay.any_glass != 0, ds.lay.n_sph, ds.lay.coord_max, ds.lay.r_min, camera);
    p.dyn_smem = p.use_smem ? smem : 0;
    return p;
}

// One-time set-up of a kernel family: the SM count, and the dynamic shared memory left next to the static arrays of its
// widest instantiation (GLASS_F64 of the first row), opted in for its instantiations that stage the scene (`staged`: rows
// indexed by GlassMode).  Each family has its own limit: K1's static arrays are larger than the adaptive kernel's.
template <typename K>
cudaError_t setup_family(std::initializer_list<const K*> staged, int& sm_count, int& dyn_limit) {
    int dev = 0, optin = 0;
    cudaFuncAttributes fa;
    cudaError_t e;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, staged.begin()[0][GLASS_F64])) != cudaSuccess) return e;
    dyn_limit = std::min(kSmemLimit, optin - (int)fa.sharedSizeBytes - 1024);
    for (const K* row : staged)
        for (int gm = GLASS_NONE; gm <= GLASS_F64; gm++)
            if ((e = cudaFuncSetAttribute(row[gm], cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit)) != cudaSuccess) return e;
    return cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
}

}  // namespace

}  // namespace rm
