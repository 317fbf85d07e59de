// rm_area.cu -- the spherical area lights' kernel (rm_render_area_lights, include/rm_b200.h RmAreaLights) and its launcher.  A
// translation unit of its own, like rm_lens.cu: instantiated next to K1 and the adaptive sub-pixel kernel it would change how
// the compiler optimises their shared inline code, and with it their machine code.
#include "rm_fast_setup.cuh"

namespace rm {

namespace {

// ---- Spherical area lights (rm_render_area_lights) ------------------------------------------------------------------------
// Primary visibility does not depend on the lights, so every pixel's primary hit is K1's, bit for bit: the same device
// functions over the raster records K0 wrote for this camera (primary_begin, primary_tri after the exact bound tri_may_touch,
// primary_rest; or primary_bvh).  Only the shading differs: fast_shade runs on an AreaView, whose direct() traces s^2 shadow
// rays per area light.
// Persistent grid.  A warp draws runs of 32 consecutive pixels of the call's n_px (rows from fp.row_begin, W-wide: a run is
// 32 pixels of one row, W being a multiple of 32) from the 64-bit counter *next (zero at launch).  Stage A runs one pixel
// per lane and stores the primary id; misses are stored black at once (renderer.rs:300-306).  Hits go to the warp's queue,
// compacted with ballot / popc, and are shaded 32 at a time on full warps; the last partial round runs when the work has run
// out.  The channel maximum of the stored values goes to *dmax.
constexpr int kAreaQueue = 64;
template <bool kSmem, bool kBvh, int kGlass>
__global__ void __launch_bounds__(kFastBlock, RM_K1_MIN_BLOCKS)
area_light_kernel(const DeviceScene<float> ds, const FrameParams<float> fp, const AreaLights al, const int cull, const long long n_px,
                  unsigned long long* __restrict__ next, float* __restrict__ rgb, int* __restrict__ prim_id, float* __restrict__ dmax,
                  const int stage_mat) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    __shared__ float4 queue[kFastBlock / 32][kAreaQueue];          // {t, slot, id, pixel of the call}
    const BlobLayout& L = ds.lay;
    const int n_tri = tri_count(L, cull != 0);
    const unsigned char* base = ds.blob;
    const R4<float>* tri_r = ds.tri_r;
    if (kSmem) {                                                // as the adaptive kernel: K0 has retired before
        stage_static(ds, stage_mat, smem_raw);
        stage_raster(ds, n_tri, smem_raw, base, tri_r);
    }
    __syncthreads();
    FastViewT<kBvh, false> fv = make_fast_view<kBvh, false>(ds, base, tri_r, n_tri, cull, kSmem && stage_mat, smem_raw);
    const AreaView<FastViewT<kBvh, false>> av(fv, al);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lane_lt = (1u << lane) - 1u;
    const bool rest = fv.n_sph + fv.n_poly > 0;
    float4* const wq = queue[warp];
    int qn = 0;                                                 // entries in this warp's queue (warp-uniform)
    float m = 0.f;
    auto shade_entry = [&](const float4 e) {
        const long long g = (long long)__float_as_uint(e.w);
        const int row = (int)(g / fp.width);
        const int x = (int)(g - (long long)row * fp.width), y = fp.row_begin + row;
        RM_CHECK(g < n_px && y < fp.row_end);
        const Vec3<float> c = fast_shade<kGlass>(av, fp, x, y, e.x, __float_as_int(e.y), __float_as_int(e.z));
        float* dst = rgb + 3 * g;
        dst[0] = c.x;
        dst[1] = c.y;
        dst[2] = c.z;
        m = fmaxf(m, fmaxf(fmaxf(c.x, c.y), c.z));
    };
    for (;;) {
        unsigned long long g0 = 0;
        if (lane == 0) g0 = atomicAdd(next, 32ull);
        g0 = __shfl_sync(0xffffffffu, g0, 0);
        if (g0 >= (unsigned long long)n_px) break;
        const long long g = (long long)g0 + lane;               // n_px is a multiple of 32: every lane is live
        const int row = (int)(g / fp.width);
        const int x = (int)(g - (long long)row * fp.width), y = fp.row_begin + row;
        PrimaryState<1> ps;
        primary_begin<1>(ps, fp, x, y);
        if constexpr (kBvh) {
            primary_bvh<1, false>(ps, fv, fp);
        } else {
            // the warp's 32 pixels: [x - lane, x - lane + 31] of row y
            const int xa = x - lane;
            const float Xa = pixel_X(fp, xa), Xb = pixel_X(fp, xa + 31), Ya = pixel_Y(fp, y), Yb = Ya;
            for (int jb = 0; jb < n_tri; jb += 32) {
                const int j = jb + lane;
                bool cand = false;
                if (j < n_tri) cand = tri_may_touch(tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], Xa, Xb, Ya, Yb);
                unsigned cm = __ballot_sync(0xffffffffu, cand);
                while (cm) {                                    // uniform across the warp
                    const int jj = jb + __ffs(cm) - 1;
                    cm &= cm - 1;
                    primary_tri<1>(ps, tri_r[4 * jj], tri_r[4 * jj + 1], tri_r[4 * jj + 2], tri_r[4 * jj + 3], fv.n_sph + jj);
                }
            }
            if (rest) primary_rest<1>(ps, fv, fp);
        }
        if (prim_id) prim_id[g] = ps.id[0];
        const bool hit = ps.slot[0] >= 0;
        if (!hit) {                                             // renderer.rs:300-306: a primary miss is black
            float* dst = rgb + 3 * g;
            dst[0] = 0.f;
            dst[1] = 0.f;
            dst[2] = 0.f;
        }
        const unsigned mh = __ballot_sync(0xffffffffu, hit);
        RM_CHECK(qn + __popc(mh) <= kAreaQueue);
        if (hit) wq[qn + __popc(mh & lane_lt)] = make_float4(ps.t[0], __int_as_float(ps.slot[0]), __int_as_float(ps.id[0]), __uint_as_float((unsigned)g));
        qn += __popc(mh);
        __syncwarp();
        if (qn >= 32) {
            qn -= 32;
            shade_entry(wq[qn + lane]);
            __syncwarp();                                       // reads done before the next round appends
        }
    }
    if (lane < qn) shade_entry(wq[lane]);
    __syncwarp();
    // values are >= 0, so the integer order of the bit patterns is the float order
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomic_max_nonneg(dmax, __int_as_float(wm));
}

}  // namespace

cudaError_t launch_area_lights(const DeviceScene<float>& ds, const FrameParams<float>& fp, const AreaLights& al, bool cull, long long n_px,
                               unsigned long long* next, float* rgb, int* prim_id, float* dmax, const double camera[3], cudaStream_t stream) {
    using K = decltype(&area_light_kernel<true, false, GLASS_NONE>);
    static const K table[3][3] = {
        {area_light_kernel<true, false, GLASS_NONE>, area_light_kernel<true, false, GLASS_F32>, area_light_kernel<true, false, GLASS_F64>},
        {area_light_kernel<false, false, GLASS_NONE>, area_light_kernel<false, false, GLASS_F32>, area_light_kernel<false, false, GLASS_F64>},
        {area_light_kernel<false, true, GLASS_NONE>, area_light_kernel<false, true, GLASS_F32>, area_light_kernel<false, true, GLASS_F64>}};
    static int sm_count = 0, dyn_limit = 0;
    cudaError_t e;
    if (!sm_count && (e = setup_family<K>({table[0]}, sm_count, dyn_limit)) != cudaSuccess) return e;
    if (n_px <= 0) return cudaSuccess;
    const FastPlan plan = fast_plan(ds, fp, camera, dyn_limit);        // K1's plan for this scene and camera
    const K k = table[plan.row()][plan.glass];
    int occ = 1;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kFastBlock, plan.dyn_smem)) != cudaSuccess) return e;
    k<<<sm_count * std::max(occ, 1), kFastBlock, plan.dyn_smem, stream>>>(ds, fp, al, cull ? 1 : 0, n_px, next, rgb, prim_id, dmax,
                                                                          plan.stage_mat);
    return cudaGetLastError();
}

}  // namespace rm
