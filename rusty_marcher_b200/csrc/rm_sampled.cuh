// rm_sampled.cuh -- the sampled-frame kernel and its launcher, one template over the effect type E: the thin-lens camera
// (rm_lens.cu), rough glass (rm_rough.cu), motion blur (rm_motion.cu), distributed ray tracing (rm_distributed.cu), diffuse
// interreflection (rm_indirect.cu) and path-traced frames (rm_path.cu).  Each of those translation units defines its E and
// instantiates the kernel for it alone: instantiated next to each other, or next to K1 and the adaptive sub-pixel kernel, the
// families would change how the compiler optimises their shared inline code, and with it their machine code.
// The shared code is the __global__ template itself: a __device__ body behind per-family kernels compiles to other code.
#pragma once

#include "rm_fast_setup.cuh"

#include <type_traits>

namespace rm {

namespace {

// What an effect type E gives the kernel:
//   E::query(fv, eff, s, r, o, d, h, st)           the level-1 closest-hit query of ray r of the item (o, d)
//   E::shade<kGlass>(fv, fp, eff, s, r, o, d, h)   the colour of that ray, whose query found h
//   E::kNoneSlot                                   the glass mode instantiated in the GLASS_NONE slot of the kernel table
// s is the lens's samples; ray r of the item is sample q = r mod s^2 of its pixel.  eff holds the effect's device arguments.
// Each E is the Effect of a namespace named after the family's kernel (lens_kernel, rough_glass_kernel, motion_kernel,
// distributed_kernel, indirect_kernel, path_kernel), so that the kernel's name in profiler output, sampled_kernel<...
// lens_kernel::Effect ...>, still holds that name.
//
// Every sample ray is the thin-lens camera's (lens_ray) and starts at a point of the lens, not at the camera, so K0's raster
// records do not apply: every ray takes a general closest-hit query from level 1 on.
// Persistent grid.  A warp draws work items from the 64-bit counter *next (zero at launch): item k is the output pixels
// [k P, k P + P) of the call's n_px pixels (rows from fp.row_begin, W-wide), P = max(kSampledRays / s^2, 1).  Ray r of the item
// is sample (i, j) = (q / s, q mod s), q = r mod s^2, of its pixel r / s^2, and 32 rays go to the warp's lanes at a time.
// Hits go to the warp's queue, compacted with ballot / popc, and are shaded 32 at a time; misses are black (renderer.rs:
// 300-306).  Every sample value lands in the warp's slice of shared memory, in resolve_box's order; once the item's queue is
// drained each of its pixels is resolved by one lane, stored, and folded into the maximum.
constexpr int kSampledRays = 128;                               // sample values per warp: 1.5 KB of shared memory
constexpr int kSampledQueue = 64;
template <typename E, bool kSmem, bool kBvh, int kGlass>
__global__ void __launch_bounds__(kFastBlock, RM_K1_MIN_BLOCKS)
sampled_kernel(const DeviceScene<float> ds, const FrameParams<float> fp, const LensCamera lc, const int cull, const long long n_px,
               unsigned long long* __restrict__ next, float* __restrict__ rgb, float* __restrict__ dmax, const int stage_mat,
               const E eff) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    __shared__ float4 queue[kFastBlock / 32][kSampledQueue];       // {t, slot, id, ray of the item}
    __shared__ float vals[kFastBlock / 32][3 * kSampledRays];
    const BlobLayout& L = ds.lay;
    const int n_tri = tri_count(L, cull != 0);
    const unsigned char* base = ds.blob;
    if (kSmem) {                                                // blob and materials (the raster records' room stays unused)
        stage_static(ds, stage_mat, smem_raw);
        base = smem_raw;
    }
    __syncthreads();
    FastViewT<kBvh, false> fv = make_fast_view<kBvh, false>(ds, base, ds.tri_r, n_tri, cull, kSmem && stage_mat, smem_raw);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lane_lt = (1u << lane) - 1u;
    const int s = lc.samples, ss = s * s;
    const int per_item = max(kSampledRays / ss, 1);
    const unsigned long long n_items = (unsigned long long)((n_px + per_item - 1) / per_item);
    float4* const wq = queue[warp];
    float* const wv = vals[warp];
    float m = 0.f;
    auto ray_of = [&](const long long p0, const int r, Vec3<double>& o, Vec3<double>& d) {
        const int q = r % ss;
        const long long p = p0 + r / ss;
        const int row = (int)(p / fp.width);
        lens_ray(lc, (int)(p - (long long)row * fp.width), fp.row_begin + row, q / s, q % s, o, d);
    };
    auto shade_entry = [&](const long long p0, const float4 e) {
        const int r = __float_as_int(e.w);
        Vec3<double> o, d;
        ray_of(p0, r, o, d);
        HitRec<float> h;
        h.dist = e.x;
        h.slot = __float_as_int(e.y);
        h.id = __float_as_int(e.z);
        const Vec3<float> c = E::template shade<kGlass>(fv, fp, eff, s, r, o, d, h);
        wv[3 * r] = c.x;
        wv[3 * r + 1] = c.y;
        wv[3 * r + 2] = c.z;
    };
    auto resolve = [&](auto tag, const int k, float (&out)[3]) {
        constexpr int S = decltype(tag)::value;
        resolve_box<S>([&](int i, float (&row)[3 * S]) {
#pragma unroll
            for (int c = 0; c < 3 * S; c++) row[c] = wv[3 * (k * S * S + i * S) + c];
        }, out);
    };
    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(next, 1ull);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const long long p0 = (long long)item * per_item;
        const int n_here = (int)min((long long)per_item, n_px - p0), n_rays = n_here * ss;
        int qn = 0;                                             // entries in this warp's queue (warp-uniform)
        for (int r0 = 0; r0 < n_rays; r0 += 32) {
            const int r = r0 + lane;
            bool hit = false;
            HitRec<float> h;
            if (r < n_rays) {
                Vec3<double> o, d;
                ray_of(p0, r, o, d);
                Counters<false> st;
                hit = E::query(fv, eff, s, r, o, d, h, st);     // renderer.rs:266
                if (!hit) {
                    wv[3 * r] = 0.f;
                    wv[3 * r + 1] = 0.f;
                    wv[3 * r + 2] = 0.f;
                }
            }
            const unsigned mh = __ballot_sync(0xffffffffu, hit);
            RM_CHECK(qn + __popc(mh) <= kSampledQueue);
            if (hit) wq[qn + __popc(mh & lane_lt)] = make_float4(h.dist, __int_as_float(h.slot), __int_as_float(h.id), __int_as_float(r));
            qn += __popc(mh);
            __syncwarp();
            if (qn >= 32) {
                qn -= 32;
                shade_entry(p0, wq[qn + lane]);
                __syncwarp();                                   // reads done before the next round appends
            }
        }
        if (lane < qn) shade_entry(p0, wq[lane]);
        __syncwarp();                                           // every sample value of the item is in wv
        for (int k = lane; k < n_here; k += 32) {
            float o[3];
            switch (s) {
                case 1: resolve(std::integral_constant<int, 1>(), k, o); break;
                case 2: resolve(std::integral_constant<int, 2>(), k, o); break;
                case 3: resolve(std::integral_constant<int, 3>(), k, o); break;
                case 4: resolve(std::integral_constant<int, 4>(), k, o); break;
                case 5: resolve(std::integral_constant<int, 5>(), k, o); break;
                case 6: resolve(std::integral_constant<int, 6>(), k, o); break;
                case 7: resolve(std::integral_constant<int, 7>(), k, o); break;
                default: resolve(std::integral_constant<int, 8>(), k, o); break;
            }
            float* dst = rgb + 3 * (p0 + k);
            dst[0] = o[0];
            dst[1] = o[1];
            dst[2] = o[2];
            m = fmaxf(m, fmaxf(fmaxf(o[0], o[1]), o[2]));
        }
        __syncwarp();                                           // resolved before the next item's values overwrite wv
    }
    // values are >= 0, so the integer order of the bit patterns is the float order
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomic_max_nonneg(dmax, __int_as_float(wm));
}

// sampled_kernel<E> over the n_px output pixels.  The ray origins leave the camera by up to the aperture, and the primitives
// may reach up to `reach` beyond their uploaded pose (0 where nothing moves): the glass mode sees the camera's extent and the
// scene's coordinates widened by them.
template <typename E>
cudaError_t launch_sampled(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const E& eff,
                           const double reach, const bool cull, const long long n_px, unsigned long long* next, float* rgb,
                           float* dmax, cudaStream_t stream) {
    // rows indexed by GlassMode, as setup_family wants them
    constexpr int kNone = E::kNoneSlot;
    using K = decltype(&sampled_kernel<E, true, false, kNone>);
    static const K table[3][3] = {
        {sampled_kernel<E, true, false, kNone>, sampled_kernel<E, true, false, GLASS_F32>, sampled_kernel<E, true, false, GLASS_F64>},
        {sampled_kernel<E, false, false, kNone>, sampled_kernel<E, false, false, GLASS_F32>, sampled_kernel<E, false, false, GLASS_F64>},
        {sampled_kernel<E, false, true, kNone>, sampled_kernel<E, false, true, GLASS_F32>, sampled_kernel<E, false, true, GLASS_F64>}};
    static int sm_count = 0, dyn_limit = 0;
    cudaError_t e;
    if (!sm_count && (e = setup_family<K>({table[0]}, sm_count, dyn_limit)) != cudaSuccess) return e;
    if (n_px <= 0) return cudaSuccess;
    const double extent[3] = {fabs(lc.cam[0]) + lc.aperture, fabs(lc.cam[1]) + lc.aperture, fabs(lc.cam[2]) + lc.aperture};
    DeviceScene<float> dm = ds;
    dm.lay.coord_max += reach;
    const FastPlan plan = fast_plan(dm, fp, extent, dyn_limit);
    const K k = table[plan.row()][plan.glass];
    int occ = 1;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kFastBlock, plan.dyn_smem)) != cudaSuccess) return e;
    k<<<sm_count * std::max(occ, 1), kFastBlock, plan.dyn_smem, stream>>>(ds, fp, lc, cull ? 1 : 0, n_px, next, rgb, dmax,
                                                                          plan.stage_mat, eff);
    return cudaGetLastError();
}

}  // namespace

}  // namespace rm
