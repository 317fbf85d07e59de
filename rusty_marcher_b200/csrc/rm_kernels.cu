// rm_kernels.cu -- hand-written sm_100a kernels of the render hot path.
//
// K1 render_kernel   replaces the Rayon loop over 32x32 patches and everything under it:
//                    engine/src/renderer.rs:63-89,128-309, shapes.rs:92-143, sphere.rs:27-61,
//                    triangle.rs:49-83, polygon.rs:60-98, obj.rs:186-216, optics.rs:4-89.
//                    One thread per pixel, a warp owns an 8x4 pixel tile, a CTA a 32x8 tile (so a
//                    reference patch is four CTAs and tile edges coincide with patch edges).  The
//                    scene's hot blob is staged once per CTA into shared memory with 128-bit
//                    copies and every lane of a warp reads the same primitive (broadcast, no bank
//                    conflicts).  The per-CTA channel maximum needed by FrameBuffer::normalize
//                    (framebuffer.rs:58-69) is fused in: warp shuffle -> shared -> one atomicMax.
// K4 tonemap_kernel  FrameBuffer::normalize + to_vec + quantize (framebuffer.rs:40-82): 16 values
//                    per thread, 128-bit loads, one 128-bit store of packed RGB8.
// ffma_probe         measures the FP32 FMA issue peak that the roofline fraction is quoted against.
//
// No tensor cores: the work is ray/primitive predicates and shading, not a dense contraction.
// Compiled with -fmad=false: FP32 code states its FMAs explicitly (rm_math.cuh), FP64 code must not
// fuse at all to stay bit-faithful to the reference.
#include "rm_kernels.h"

#include <algorithm>
#include <cassert>
#include <cstdlib>

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

constexpr int kBlock = 256;          // 8 warps: 4 across x 2 down, each an 8x4 pixel tile
constexpr int kTileW = 32, kTileH = 8;
constexpr int kSmemLimit = 200 * 1024;

template <typename R>
__device__ __forceinline__ SceneView<R> make_view(const DeviceScene<R>& ds, const unsigned char* base, int cull) {
    SceneView<R> sc;
    const BlobLayout& L = ds.lay;
    sc.sph = reinterpret_cast<const R4<R>*>(base + L.off_sph);
    sc.sph_id = reinterpret_cast<const int*>(base + L.off_sph_id);
    sc.n_sph = L.n_sph;
    sc.pln_n = reinterpret_cast<const R4<R>*>(base + L.off_pln_n);
    sc.pln_c = reinterpret_cast<const R4<R>*>(base + L.off_pln_c);
    sc.pln_v = reinterpret_cast<const I2*>(base + L.off_pln_v);
    sc.pln_id = reinterpret_cast<const int*>(base + L.off_pln_id);
    sc.n_pln = plane_count<R>(L, cull != 0);
    sc.vert = reinterpret_cast<const VertT<R>*>(base + L.off_vert);
    sc.mat_a = ds.mat_a;
    sc.mat_b = ds.mat_b;
    sc.mat_f = ds.mat_f;
    sc.lgt_p = reinterpret_cast<const R4<R>*>(base + L.off_lgt_p);
    sc.lgt_c = reinterpret_cast<const R4<R>*>(base + L.off_lgt_c);
    sc.n_lgt = L.n_lgt;
    sc.order = ds.order[cull];
    sc.order_shape = ds.order_shape[cull];
    sc.n_order = ds.n_order[cull];
    return sc;
}

__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));            // v >= 0: int order == float order
}
__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v) {
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// ---- programmatic dependent launch: the render kernel is launched while the prepare kernel (K0) still runs; its CTAs
// become resident, stage the static scene into shared memory and then wait here for K0's results (raster records, tile
// schedule, zeroed maximum) -- the launch latency and the prologue of K1 hide behind K0.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_primary() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- peer-memory exchange (PeerLink, rm_kernels.h): system-scope words in mailboxes every GPU of the box has mapped ----
constexpr unsigned long long kPeerTimeoutNs = 2000000000ull;    // a wait gives up after 2 s (a peer died): flag it, go on
__device__ __forceinline__ unsigned long long ld_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Spins until the upper half of *p is `seq`; returns the word.
__device__ __noinline__ unsigned long long wait_word(const unsigned long long* p, const unsigned seq, unsigned long long* err) {
    unsigned long long v = ld_sys(p);
    if ((unsigned)(v >> 32) == seq) return v;
    const unsigned long long t0 = now_ns();
    for (int spins = 0;; spins++) {
        v = ld_sys(p);
        if ((unsigned)(v >> 32) == seq) return v;
        if (spins > 64) __nanosleep(64);
        if ((spins & 1023) == 1023 && now_ns() - t0 > kPeerTimeoutNs) {
            st_sys(err, ((unsigned long long)seq << 32) | 1ull);
            return v;
        }
    }
}
// Render kernel, last CTA out: this rank's channel maximum of frame link.seq to every rank's mailbox (its own included).
__device__ __forceinline__ void publish_max(const PeerLink& link, const float m) {
    RM_CHECK(link.world >= 1 && link.world <= kMaxRanks && link.rank >= 0 && link.rank < link.world && link.seq != 0u && m >= 0.f);
    const unsigned long long w = ((unsigned long long)link.seq << 32) | (unsigned long long)__float_as_uint(m);
    for (int r = 0; r < link.world; r++) st_sys(link.box[r] + (link.seq & 1u) * 16 + link.rank, w);
}
// Tone-map kernels, every block: the frame's maximum = max over the ranks' published words (FrameBuffer::normalize is a
// global maximum, framebuffer.rs:58-69).  Lane r of warp 0 waits for rank r's word.
__device__ __forceinline__ float gather_max(const PeerLink& link, float* slot) {
    if (threadIdx.x < 32) {
        float m = 0.f;
        unsigned long long* mine = link.box[link.rank];
        if ((int)threadIdx.x < link.world)
            m = __uint_as_float((unsigned)wait_word(mine + (link.seq & 1u) * 16 + threadIdx.x, link.seq, mine + 48));
        m = __int_as_float(__reduce_max_sync(0xffffffffu, __float_as_int(m)));     // values >= 0: int order == float order
        if (threadIdx.x == 0) *slot = m;
    }
    __syncthreads();
    return *slot;
}
// Tone-map kernels, after a block's last store: the last block of the grid to get here tells rank 0 that this rank's
// bytes of the frame are in place; on rank 0 it waits for everybody else's signal, so the kernel retires with the whole
// frame assembled.  `done` is a zero-initialised local counter, left at zero.
__device__ __forceinline__ void signal_frame_done(const PeerLink& link, int* done) {
    __syncthreads();
    if (threadIdx.x != 0 || link.world < 1) return;
    // This block's stores (peer memory included) are ordered before its count by a device-scope fence; the one system-
    // scope fence of the last block then covers them all (fences are cumulative) -- a fence.sys per block costs ~5 us.
    __threadfence();
    if (atomicAdd(done, 1) != (int)gridDim.x - 1) return;
    *done = 0;
    link.box[link.rank][59] = now_ns();                        // stamp: this rank's bytes stored
    if (link.world == 1) return;
    __threadfence_system();
    if (link.rank != 0) {
        st_sys(link.box[0] + 32 + link.rank, ((unsigned long long)link.seq << 32) | 1ull);
    } else {
        for (int r = 1; r < link.world; r++) wait_word(link.box[0] + 32 + r, link.seq, link.box[0] + 48);
        __threadfence_system();
        link.box[0][60] = now_ns();                            // stamp: frame complete on rank 0
    }
}

template <typename R> struct Tone;
template <> struct Tone<float> {
    static __device__ __forceinline__ unsigned q(float v, float inv) {
        return (unsigned)(unsigned char)(255.f * fminf(fmaxf(v * inv, 0.f), 1.f));     // framebuffer.rs:80-82
    }
};
template <> struct Tone<double> {
    static __device__ __forceinline__ unsigned q(double v, double inv) {
        return (unsigned)(unsigned char)(255. * fmin(fmax(v * inv, 0.), 1.));
    }
};

template <typename R, bool S>
__global__ void __launch_bounds__(kBlock)
render_kernel(const DeviceScene<R> ds, const FrameParams<R> fp, const int cull, const int use_smem,
              R* __restrict__ rgb, int* __restrict__ prim_id, R* __restrict__ dmax,
              unsigned long long* __restrict__ counters) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    __shared__ R warp_max[kBlock / 32];

    const unsigned char* base = ds.blob;
    if (use_smem) {
        const uint4* src = reinterpret_cast<const uint4*>(ds.blob);
        uint4* dst = reinterpret_cast<uint4*>(smem_raw);
        for (int i = threadIdx.x; i < ds.lay.bytes / 16; i += kBlock) dst[i] = __ldg(src + i);
        __syncthreads();
        base = smem_raw;
    }
    const SceneView<R> sc = make_view<R>(ds, base, cull);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int x = blockIdx.x * kTileW + (warp & 3) * 8 + (lane & 7);
    const int yl = blockIdx.y * kTileH + (warp >> 2) * 4 + (lane >> 3);   // row within this call's bands
    const int y = frame_row(fp, yl);

    Counters<S> st;
    st.clear();

    R m = R(0);
    if (x < fp.width && yl < fp.n_bands * 32) {
        st.add(C_PIXELS);
        int pid;
        const Vec3<R> dir = backproject<R>(fp, x, y);
        const Vec3<R> c = cast_ray<R, S, SceneView<R>>(sc, fp.camera, dir, fp.background, fp.max_depth, pid, st);
        const size_t px = (size_t)(y - fp.buf_row0) * fp.width + x;
        rgb[3 * px] = c.x;
        rgb[3 * px + 1] = c.y;
        rgb[3 * px + 2] = c.z;
        if (prim_id) prim_id[px] = pid;
        m = Num<R>::max_(Num<R>::max_(Num<R>::max_(c.x, c.y), c.z), R(0));
    }

    // fused K3: channel maximum of the tile (framebuffer.rs:58-69)
    for (int off = 16; off > 0; off >>= 1) m = Num<R>::max_(m, __shfl_xor_sync(0xffffffffu, m, off));
    if (lane == 0) warp_max[warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kBlock / 32; w++) m = Num<R>::max_(m, warp_max[w]);
        if (m > R(0)) atomic_max_nonneg(dmax, m);
    }

    if (S) {
        const unsigned* c = reinterpret_cast<const unsigned*>(&st);
        for (int i = 0; i < C_COUNT; i++) {
            unsigned v = c[i];
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0 && v) atomicAdd(counters + i, (unsigned long long)v);
        }
    }
}

// K0: camera-specialised raster records of every fast-path triangle, in FP64, once per frame.
__global__ void __launch_bounds__(128)
prepare_raster_kernel(const double* __restrict__ tri_src, const int n_tri, const double cx, const double cy, const double cz,
                      R4<float>* __restrict__ tri_r, float* __restrict__ dmax_zero) {
    pdl_launch_dependents();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j == 0 && dmax_zero) *dmax_zero = 0.f;
    if (j >= n_tri) return;
    const double cam[3] = {cx, cy, cz};
    R4<float> out[4];
    prepare_raster(tri_src + (size_t)j * kTriSrcDoubles, cam, out);
#pragma unroll
    for (int k = 0; k < 4; k++) tri_r[4 * j + k] = out[k];
}

// K0 for scenes made of (few) triangles only: the raster records as above, and in the same launch the
// tile schedule of the render kernel.  Eight lanes per 32x32 tile bound the triangles against the tile, one
// triangle per lane and round (tri_may_touch: exact, see rm_fast.cuh); tiles some triangle may touch are "busy" and go to the front of
// the schedule, the others are provably black and go to the back.  The render kernel hands the busy
// tiles out first (longest work first, so the cheap tiles fill the tail) and only stores zeros for the rest.
// (K0 was also tried fused into the render kernel behind a grid-wide barrier: 4.2 us inside the kernel -- the barrier
// exposes the launch ramp of the 296 CTAs -- against 2.3 us of K0 plus a 3 to 4.6 us hand-over here, whose first part
// overlaps K1's launch thanks to the programmatic dependent launch.  No gain; not kept.)
constexpr int kClassifyMaxTris = 256;
constexpr int kClassifyBlock = 512, kClassifyLanes = 8;         // 8 lanes per tile: 64 tiles per block
__global__ void __launch_bounds__(kClassifyBlock)
prepare_classify_kernel(const double* __restrict__ tri_src, const int n_tri, const double cx, const double cy, const double cz,
                        R4<float>* __restrict__ tri_r, const FrameParams<float> fp, const int tiles_x, const int n_tiles,
                        int* __restrict__ order, int* __restrict__ order2, int* __restrict__ ctr, float* __restrict__ dmax_zero) {
    __shared__ R4<float> rec[4 * kClassifyMaxTris];
    __shared__ int cnt[3], base[3];
    const double cam[3] = {cx, cy, cz};
    pdl_launch_dependents();
    unsigned long long* const stamp = reinterpret_cast<unsigned long long*>(ctr + 12);   // [0] K0 start, [1] K0 end (ns)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (dmax_zero) *dmax_zero = 0.f;
        stamp[0] = now_ns();
        stamp[1] = 0ull;
    }
    if (threadIdx.x < 3) cnt[threadIdx.x] = 0;
    for (int j = threadIdx.x; j < n_tri; j += blockDim.x) {      // every block rebuilds the (few) records; block 0 publishes them
        R4<float> out[4];
        prepare_raster(tri_src + (size_t)j * kTriSrcDoubles, cam, out);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            rec[4 * j + k] = out[k];
            if (blockIdx.x == 0) tri_r[4 * j + k] = out[k];
        }
    }
    __syncthreads();
    // a tile is tested by kClassifyLanes lanes, lane s against triangles s, s + 8, ...; the group's verdict is read off a ballot
    const int lane = threadIdx.x & 31, sub = lane & (kClassifyLanes - 1);
    const int tile = (blockIdx.x * kClassifyBlock + threadIdx.x) / kClassifyLanes;
    bool touch = false, cover = false;
    if (tile < n_tiles) {
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        const int x0 = tx * 32, y0 = fp.row_begin + ty * fp.row_step;
        const float Xa = pixel_X(fp, x0), Xb = pixel_X(fp, x0 + 31), Ya = pixel_Y(fp, y0), Yb = pixel_Y(fp, y0 + 31);
        for (int j = sub; j < n_tri && !cover; j += kClassifyLanes) {
            if (tri_may_touch(rec[4 * j], rec[4 * j + 1], rec[4 * j + 2], rec[4 * j + 3], Xa, Xb, Ya, Yb)) {
                touch = true;
                cover = tri_covers(rec[4 * j], rec[4 * j + 1], rec[4 * j + 2], rec[4 * j + 3], Xa, Xb, Ya, Yb);
            }
        }
    }
    const unsigned group = ((1u << kClassifyLanes) - 1u) << (lane & ~(kClassifyLanes - 1));
    const bool busy = (__ballot_sync(0xffffffffu, touch) & group) != 0u;
    const bool full = (__ballot_sync(0xffffffffu, cover) & group) != 0u;
    // Three classes: fully covered tiles (1024 hits to shade: the longest jobs) at the front of `order`, partially covered
    // ones in `order2` (handed out after the full ones), empty ones from the back of `order`.  The group leaders take a
    // place within the block from shared counters; three global atomics per block reserve the block's ranges.
    const bool leader = sub == 0 && tile < n_tiles;
    const int cls = full ? 0 : busy ? 1 : 2;
    int local = 0;
    if (leader) local = atomicAdd(&cnt[cls], 1);
    __syncthreads();
    if (threadIdx.x < 3 && cnt[threadIdx.x]) base[threadIdx.x] = atomicAdd(ctr + (threadIdx.x == 0 ? 1 : threadIdx.x == 1 ? 5 : 2), cnt[threadIdx.x]);
    __syncthreads();
    if (leader) {
        if (cls == 0) order[base[0] + local] = tile;
        else if (cls == 1) order2[base[1] + local] = tile;
        else order[n_tiles - 1 - (base[2] + local)] = tile;
    }
    if (threadIdx.x == 0) atomicMax(stamp + 1, now_ns());
}

// K1, FP32 production kernel (rm_fast.cuh).  Persistent and warp-granular: the grid is (SMs x resident
// CTAs); every CTA stages the scene into shared memory ONCE; after that its warps never meet at a
// barrier again.  Work is handed out per WARP, the GPU analogue of Rayon's work stealing over the
// reference's 32x32 patches (renderer.rs:46-89) at a granularity that suits 3552 resident warps: a warp
// draws one 32x4 strip (an eighth of a patch) at a time from a global atomic counter that walks the tile
// schedule, fully covered tiles first.  (Handing whole tiles to CTAs quantised the kernel's duration to
// ceil(busy tiles / CTAs) tile times: 3 rounds instead of 2.7 on the cornell frame, and no gain at all
// from splitting the frame over two GPUs.)
// Per strip a warp runs a two-stage wavefront of its own:
//   A  primary visibility, divergence-free: a thread owns 4 horizontally adjacent pixels.  First the
//      warp bounds every triangle against the strip (one triangle per lane, exact corner test
//      tri_may_touch, ballot), then all lanes walk the surviving triangles together (primary_tri<4>).
//      Misses are final (black) and are written at once with 128-bit stores; hits are appended to the
//      warp's private shared-memory queue, compacted with ballot/popc, so that
//   B  shading + shadow rays + the reflect/refract recursion (the divergent part) runs on a fully
//      populated warp: whenever the queue holds 32 entries or more, one entry per lane.  A remainder
//      waits for the next strip's hits; when the busy tiles have run out the warps first zero-fill the
//      tiles the classify kernel proved empty (drawn per warp, nothing to balance), then pool their
//      leftovers across the CTA for one last round on full warps.
// The channel maximum (framebuffer.rs:58-69) is kept per thread across all its strips and reduced once:
// REDUX over the warp, shared atomic, one global atomic per CTA.
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
constexpr int kFastTile = 32;
constexpr int kWarpQueue = kFastTile * 4 + 32;                  // one strip of hits on top of a partial round
#ifdef RM_K1_MAXREG
#define RM_K1_BOUNDS __maxnreg__(RM_K1_MAXREG)
#else
#define RM_K1_BOUNDS __launch_bounds__(kFastBlock, kGlass != GLASS_NONE ? RM_K1_MIN_BLOCKS : RM_K1_MIN_BLOCKS_OPAQUE)
#endif
#ifndef RM_K1_MIN_BLOCKS_OPAQUE
#define RM_K1_MIN_BLOCKS_OPAQUE 2                               // the instantiation without recursion / f64 code (kGlass = false)
#endif
template <int kPx> struct PxTag { static constexpr int value = kPx; };
// kBvh (RmParams.accel): scene queries walk the hierarchy of rm_bvh.cuh (read through the read-only path; the nodes near
// the root stay in L1) instead of every primitive; stage A then handles a thread's pixels one after the other.
template <bool kSmem, int kBvhMode, int kGlass>
__global__ void RM_K1_BOUNDS
render_fast_kernel(const DeviceScene<float> ds, const FrameParams<float> fp, const int cull, const int tiles_x,
                   const int n_tiles, const float inv_tiles_x, float* __restrict__ rgb, int* __restrict__ prim_id,
                   float* __restrict__ dmax, int* __restrict__ ctr, const int* __restrict__ order, const int* __restrict__ order2,
                   unsigned char* rgb8, const PeerLink link, unsigned char* rgb8_out, const int normalise,
                   unsigned char* rgb8_next, const int stage_mat) {
    constexpr bool kBvh = kBvhMode != 0, kCount = kBvhMode == 2;    // 2: the counting instantiation (RmParams.accel = 2)
    const int zero_foreign = rgb8_next != nullptr;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    __shared__ int cta_max;
    __shared__ float frame_max;
    __shared__ int leftover[kFastBlock / 32];
    __shared__ int fill_off[96];                                // float offset of each 16-byte chunk of a strip (see fill_strip)
    __shared__ float4 pool[kFastBlock];                             // pooled leftovers of the eight warp queues (< 32 each)
    __shared__ float4 queue[kFastBlock / 32][kWarpQueue];           // {t, slot, id, x | y << 16}
    const BlobLayout& L = ds.lay;
    const int n_tri = tri_count(L, cull != 0);

    const unsigned char* base = ds.blob;
    const R4<float>* tri_r = ds.tri_r;
    if (threadIdx.x < 96) fill_off[threadIdx.x] = (threadIdx.x / 24) * fp.width * 3 + (threadIdx.x % 24) * 4;
    if (threadIdx.x == 0) cta_max = 0;
    if (kSmem) {                                                // the static part of the scene: does not depend on K0
        const uint4* src = reinterpret_cast<const uint4*>(ds.blob);
        uint4* dst = reinterpret_cast<uint4*>(smem_raw);
        const int n16 = L.bytes / 16;
        for (int i = threadIdx.x; i < n16; i += kFastBlock) dst[i] = __ldg(src + i);
        if (stage_mat) {                                        // materials behind the raster records: mat_a | mat_b | mat_f
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
    pdl_wait_primary();                                         // K0 has retired: raster records, schedule, zeroed maximum
    if (threadIdx.x == 0 && blockIdx.x == 0 && link.world > 0) {
        unsigned long long* const box = link.box[link.rank];
        box[56] = now_ns();                                     // stamp: start of the work
        box[61] = reinterpret_cast<const unsigned long long*>(ctr + 12)[0];     // K0's own stamps, for the phase breakdown
        box[62] = reinterpret_cast<const unsigned long long*>(ctr + 12)[1];     // (tile-scheduled scenes only)
    }
    if (kSmem) {
        uint4* dst = reinterpret_cast<uint4*>(smem_raw);
        const int n16 = L.bytes / 16;
        const uint4* rsrc = reinterpret_cast<const uint4*>(ds.tri_r);
        for (int i = threadIdx.x; i < n_tri * 4; i += kFastBlock) dst[n16 + i] = rsrc[i];
        base = smem_raw;
        tri_r = reinterpret_cast<const R4<float>*>(smem_raw + L.bytes);
    }
    __syncthreads();
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
    if (kSmem && stage_mat) {
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

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lane_lt = (1u << lane) - 1u;
    const bool rest = fv.n_sph + fv.n_poly > 0;
    // schedule: [0, n_full) fully covered tiles (order), [n_full, n_busy) partially covered (order2), [n_busy, n_tiles) empty (order)
    const int n_full = order ? ctr[1] : n_tiles, n_busy = order ? n_full + ctr[5] : n_tiles;
    float4* const wq = queue[warp];
    int qn = 0;                                                 // entries in this warp's queue (warp-uniform)
    int final_take = 0;
    float m = 0.f;

    auto shade_entry = [&](const float4 e) {
        const unsigned xy = __float_as_uint(e.w);
        const int x = (int)(xy & 0xffffu), y = (int)(xy >> 16);
        const Vec3<float> c = fast_shade<kGlass>(fv, fp, x, y, e.x, __float_as_int(e.y), __float_as_int(e.z));
        RM_CHECK(x >= 0 && x < fp.width && y >= fp.row_begin && y < fp.row_begin + (fp.n_bands - 1) * fp.row_step + 32 &&
                 (y - fp.row_begin) % fp.row_step < 32);
        float* dst = rgb + 3 * ((size_t)(y - fp.buf_row0) * fp.width + x);
        dst[0] = c.x;
        dst[1] = c.y;
        dst[2] = c.z;
        m = fmaxf(m, fmaxf(fmaxf(c.x, c.y), c.z));
    };

    // Zero-fill (renderer.rs:300-306: a primary miss is black) of a 32-pixel wide strip of kStripRows rows by one warp,
    // fully coalesced: a pixel row of the strip is 384 contiguous bytes = 24 chunks of 16 bytes, the strip 96 chunks,
    // lane l stores chunks l, l + 32, l + 64 (each instruction writes 512 bytes in at most two contiguous runs).
    // With rgb8 given the strip's bytes of the 8-bit frame are zeroed as well: quantize(0 * 1/max) is 0 whatever the
    // maximum turns out to be (framebuffer.rs:71-82), so only the busy tiles are left for the tone-map kernel.  A row of
    // the strip is 96 bytes = 6 chunks of 16 bytes, the strip 24 chunks: one store of lanes 0..23.
    auto fill_rows = [&](const size_t p0, const int rows) {     // p0: pixel index of the first pixel; rows: 2 or 4
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        float* const strip0 = rgb + 3 * p0;
#pragma unroll
        for (int i = 0; i < 3; i++)
            if (lane + 32 * i < 24 * rows) __stcs(reinterpret_cast<float4*>(strip0 + fill_off[lane + 32 * i]), z);
        if (rgb8 && lane < 6 * rows) __stcs(reinterpret_cast<uint4*>(rgb8 + 3 * p0 + (size_t)(lane / 6) * fp.width * 3 + (lane % 6) * 16), make_uint4(0u, 0u, 0u, 0u));
    };
    auto fill_empty_tile = [&](const int tile) {                // always in pieces of four rows, whatever the strip height
        const int ty = (int)(((float)tile + 0.5f) * inv_tiles_x);
        const int tx = tile - ty * tiles_x;
        RM_CHECK(tile >= 0 && tile < n_tiles && ty == tile / tiles_x && tx >= 0 && tx < tiles_x && ty < fp.n_bands);
        const size_t p0 = (size_t)(fp.row_begin + ty * fp.row_step - fp.buf_row0) * fp.width + tx * kFastTile;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            fill_rows(p0 + (size_t)r * 4 * fp.width, 4);
            if (prim_id) __stcs(reinterpret_cast<int4*>(prim_id + p0 + (size_t)(r * 4 + (lane >> 3)) * fp.width + (lane & 7) * 4), make_int4(-1, -1, -1, -1));
        }
    };
    // The empty tiles' stores are pure HBM traffic and must overlap the busy tiles' arithmetic instead of forming a
    // phase of their own.  Every warp of the grid owns a fixed share of the schedule's empty part (nothing to balance:
    // tiles gw, gw + W, ... for global warp gw of W) and works it off at the pace of the busy strips it processes:
    // n_empty / n_busy_strips empty tiles per busy strip, carried in a fraction accumulator.  What is left when the busy
    // tiles run out (all of it for warps that never drew a busy strip) is filled in phase 2.
    const int n_empty = n_tiles - n_busy;
    const int n_warps_grid = gridDim.x * (kFastBlock / 32);
    // Strip height (a strip is 32 pixels wide and kPx rows high: 32 lanes x kPx horizontally adjacent pixels of a thread in
    // stage A).  Four rows amortise the record loads of stage A best, but a fully covered strip is then four shading rounds
    // in a row on one warp, and on a GPU with few strips -- its share of a frame split over several GPUs, a sparsely
    // covered frame -- the longest such chain sets the kernel's duration.  Two-row strips halve it.  Decided per launch
    // from the schedule: four rows when there are at least two fully covered four-row strips per warp of the grid.
    const bool tall = order && n_full * 8 >= 2 * n_warps_grid;
    const int n_busy_strips = n_busy * (tall ? 8 : 16);
    const int n_warps = n_warps_grid;
    int next_empty = n_busy + blockIdx.x * (kFastBlock / 32) + warp;   // schedule position of this warp's next empty tile
    int empty_acc = 0;

    auto warp_loop = [&](auto px_tag) {
    constexpr int kPx = decltype(px_tag)::value;
    constexpr int kStripRows = kPx, kStripsPerTile = kFastTile / kStripRows, kRowLanes = 32 / kPx;
    const int lx = (lane % kRowLanes) * kPx, ly = lane / kRowLanes;
    // ---- phase 1: busy tiles, dynamic.  phase 3 (below) reuses the shading code of the loop through `pooled`.
    for (int phase = 1;;) {
        if (phase == 1) {
            // next strip of the schedule: strip s & 7 of the (s >> 3)-th busy tile.  One global atomic per 128 pixels;
            // its latency hides behind the other warps of the SM, and no warp ever holds work another one could do.
            int s = 0;
            if (lane == 0) s = atomicAdd(ctr, 1);
            s = __shfl_sync(0xffffffffu, s, 0);
            const int k = s / kStripsPerTile, strip = s % kStripsPerTile;
            if (k >= n_busy) {
                phase = 2;
            } else {
                const int tile = !order ? k : k < n_full ? __ldg(order + k) : __ldg(order2 + (k - n_full));
                const int ty = (int)(((float)tile + 0.5f) * inv_tiles_x);          // exact for tile < 2^22
                const int tx = tile - ty * tiles_x;
                RM_CHECK(tile >= 0 && tile < n_tiles && ty == tile / tiles_x && tx >= 0 && tx < tiles_x && ty < fp.n_bands);
                RM_CHECK(n_full >= 0 && n_busy >= n_full && n_busy <= n_tiles);
                const int x0 = tx * kFastTile, ys = fp.row_begin + ty * fp.row_step + strip * kStripRows;
                const size_t px = (size_t)(ys + ly - fp.buf_row0) * fp.width + x0 + lx;
                fill_rows((size_t)(ys - fp.buf_row0) * fp.width + x0, kStripRows);         // misses stay black; stage B overwrites the hits
                // stage A: primary visibility of this thread's 4 pixels
                PrimaryState<kPx> ps;
                primary_begin<kPx>(ps, fp, x0 + lx, ys + ly);
                if constexpr (kBvh) {
                    primary_bvh<kPx, kCount>(ps, fv, fp);
                } else {
                    // the strip: pixels [x0, x0 + 31] x [ys, ys + 3]
                    const float Xa = pixel_X(fp, x0), Xb = pixel_X(fp, x0 + kFastTile - 1);
                    const float Ya = pixel_Y(fp, ys), Yb = pixel_Y(fp, ys + kStripRows - 1);
                    for (int jb = 0; jb < n_tri; jb += 32) {
                        const int j = jb + lane;
                        bool cand = false;
                        if (j < n_tri) cand = tri_may_touch(tri_r[4 * j], tri_r[4 * j + 1], tri_r[4 * j + 2], tri_r[4 * j + 3], Xa, Xb, Ya, Yb);
                        unsigned cm = __ballot_sync(0xffffffffu, cand);
                        while (cm) {                            // uniform across the warp
                            const int jj = jb + __ffs(cm) - 1;
                            cm &= cm - 1;
                            primary_tri<kPx>(ps, tri_r[4 * jj], tri_r[4 * jj + 1], tri_r[4 * jj + 2], tri_r[4 * jj + 3], fv.n_sph + jj);
                        }
                    }
                    if (rest) primary_rest<kPx>(ps, fv, fp);
                }
                if (prim_id) {
                    if (kPx == 4) __stcs(reinterpret_cast<int4*>(prim_id + px), make_int4(ps.id[0], ps.id[1], ps.id[kPx - 2], ps.id[kPx - 1]));
                    else __stcs(reinterpret_cast<int2*>(prim_id + px), make_int2(ps.id[0], ps.id[1]));
                }
                // hits -> the warp's queue, pixel column by pixel column, compacted with ballot / popc
                const unsigned xy = (unsigned)(x0 + lx) | ((unsigned)(ys + ly) << 16);
#pragma unroll
                for (int c = 0; c < kPx; c++) {
                    const unsigned mc = __ballot_sync(0xffffffffu, ps.slot[c] >= 0);
                    RM_CHECK(qn + __popc(mc) <= kWarpQueue);
                    if (ps.slot[c] >= 0) wq[qn + __popc(mc & lane_lt)] = make_float4(ps.t[c], __int_as_float(ps.slot[c]), __int_as_float(ps.id[c]), __uint_as_float(xy + c));
                    qn += __popc(mc);
                }
                __syncwarp();
                if (next_empty < n_tiles) {
                    empty_acc += n_empty;
                    while (empty_acc >= n_busy_strips && next_empty < n_tiles) {
                        empty_acc -= n_busy_strips;
                        fill_empty_tile(order[next_empty]);
                        next_empty += n_warps;
                    }
                }
            }
        }
        if (phase == 2) {
            // ---- phase 2: the busy tiles have run out: the rest of this warp's share of the empty tiles
            for (; next_empty < n_tiles; next_empty += n_warps) fill_empty_tile(order[next_empty]);
            // ---- phase 3: pool the warps' leftovers (< 32 each) so the last round runs on full warps again
            if (lane == 0) leftover[warp] = qn;
            __syncthreads();
            int before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < kFastBlock / 32; w++) {
                const int c = leftover[w];
                if (w < warp) before += c;
                total += c;
            }
            RM_CHECK(qn < 32 && total < kFastBlock && before + qn <= kFastBlock);
            if (lane < qn) pool[before + lane] = wq[lane];
            __syncthreads();
            final_take = min(max(total - warp * 32, 0), 32);    // total < 256: at most one round, warp w takes entries [32 w, 32 w + 32)
            phase = 3;
        }
        // ---- stage B: full warps only, from the tail of the queue (phase 3: this warp's share of the pooled leftovers)
        for (;;) {
            const float4* src;
            int take;
            if (phase == 3) {
                src = pool + warp * 32;
                take = final_take;
            } else {
                if (qn < 32) break;
                qn -= 32;
                src = wq + qn;
                take = 32;
            }
            if (lane < take) shade_entry(src[lane]);
            if (phase == 3) break;
        }
        if (phase == 3) break;
        __syncwarp();                                           // reads done before the next strip appends
    }
    };
    if (tall) warp_loop(PxTag<4>());
    else warp_loop(PxTag<2>());
    if constexpr (kBvh) {                                       // ctr[6..7]: u64 count of secondary + shadow queries, kept across frames
        const unsigned q = __reduce_add_sync(0xffffffffu, fv.n_queries);
        if (lane == 0 && q) atomicAdd(reinterpret_cast<unsigned long long*>(ctr + 6), (unsigned long long)q);
    }
    if constexpr (kCount) {                                     // status words [10..15]: three u64 (node visits, sphere tests, plane tests)
        unsigned long long* w = reinterpret_cast<unsigned long long*>(ds.bvh.status + 10);
        // (per-thread 32-bit counts summed in 64 bits: a lane of a heavy frame stays far below 2^32)
        unsigned long long a = fv.cnt.nodes, b = fv.cnt.sph, c = fv.cnt.pln;
        for (int off = 16; off > 0; off >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, off);
            b += __shfl_xor_sync(0xffffffffu, b, off);
            c += __shfl_xor_sync(0xffffffffu, c, off);
        }
        if (lane == 0) {
            atomicAdd(w, a);
            atomicAdd(w + 1, b);
            atomicAdd(w + 2, c);
        }
    }
    // values are >= 0, so the integer order of the bit patterns is the float order
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomicMax(&cta_max, wm);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (cta_max > 0) atomicMax(reinterpret_cast<int*>(dmax), cta_max);
        // the last CTA out leaves the frame control block zeroed for the next frame
        __threadfence();
        if (atomicAdd(ctr + 3, 1) == (int)gridDim.x - 1) {
            ctr[8] = order ? n_full : -1;                       // kept for the busy-tiles-only tone-map kernel of this frame
            ctr[9] = n_busy - n_full;
            ctr[0] = 0;
            ctr[1] = 0;
            ctr[2] = 0;
            ctr[3] = 0;
            ctr[5] = 0;
            // every CTA's stores and its atomicMax happened before its count (fence above): the maximum of this rank's
            // rows is final, and so are its float rows and (rank 0) the cleared bytes of the 8-bit frame
            if (link.world > 0) {
                link.box[link.rank][57] = now_ns();                                                 // stamp: rendering done
                // Rank 0's cleared bytes must be in place before a peer, having seen this word, stores its tiles over them:
                // system-scope fence (cumulative over the CTAs counted above).  Nothing a peer touches depends on the
                // other ranks' stores, and a fence.sys costs microseconds.
                if (link.world > 1 && link.rank == 0) __threadfence_system();
                publish_max(link, __int_as_float(atomicMax(reinterpret_cast<int*>(dmax), 0)));
            }
        }
    }
    if (!rgb8_out) return;
    // ---- phase 4: FrameBuffer::normalize + to_vec (framebuffer.rs:40-82), fused.  Every CTA waits for the words of all
    // ranks in this rank's mailbox -- its own word is only published once every CTA of this grid has retired from
    // rendering, so the wait is also the grid-wide barrier that makes the float rows readable (the grid is persistent:
    // all its CTAs are resident, nobody waits for a CTA that cannot start) -- takes the maximum, and converts the busy
    // tiles, one tile per CTA and round, straight into rank 0's 8-bit frame (peer memory on ranks > 0).
    float inv = 1.f;
    {
        const float mx = gather_max(link, &frame_max);
        if (normalise && mx > 0.f) inv = 1.f / mx;              // framebuffer.rs:71-76: scale(1. / max_val)
        if (blockIdx.x == 0 && threadIdx.x == 0) link.box[link.rank][58] = now_ns();                // stamp: maxima gathered
    }
    // A wait that gave up (a rank -- or, on a shared device, CTAs of this very grid -- did not answer within 2 s): the float
    // rows behind the barrier are not known to be complete.  Nothing is converted, the sticky flag (rm_peer_status) says why
    // the 8-bit frame is stale; whoever waits for this rank's signal gives up the same way.
    if (ld_sys(link.box[link.rank] + 48) != 0ull) return;
    __threadfence();
    // Work unit: a 32x4 strip of a busy tile = 96 float4 in, 24 x 16 bytes out (a row of the strip is 96 bytes of RGB8: six
    // 128-bit stores).  A warp takes four units per round and issues their twelve fully coalesced loads (lane l reads chunks
    // l, l + 32, l + 64 of a unit) before the first conversion -- the phase is bound by L2 latency, not by bytes.  A chunk
    // converts to one 4-byte word; the words of four neighbouring lanes are one aligned 16-byte piece of the 8-bit row,
    // gathered with three shuffles and stored by the first of the four: every store -- into rank 0's frame over NVLink on
    // ranks > 0 -- is a full 128-bit one.  (Letting a lane load its own four chunks instead strides the loads by 64 bytes:
    // twice the L2 sector requests, tone phase 6.2 instead of 5.2 us.)
    {
        constexpr int kToneRows = 4, kTonePerTile = kFastTile / kToneRows;
        const int n_units = n_busy * kTonePerTile;
        const int gw = blockIdx.x * (kFastBlock / 32) + warp;
        for (int u0 = gw; u0 < n_units; u0 += 4 * n_warps) {
            float4 q[4][3];
            size_t base_v[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int u = u0 + k * n_warps;
                base_v[k] = 0;
                if (u < n_units) {
                    const int t = u / kTonePerTile, strip = u - t * kTonePerTile;
                    const int tile = !order ? t : t < n_full ? __ldg(order + t) : __ldg(order2 + (t - n_full));
                    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
                    RM_CHECK(tile >= 0 && tile < n_tiles && ty < fp.n_bands);
                    base_v[k] = 3 * ((size_t)(fp.row_begin + ty * fp.row_step + strip * kToneRows - fp.buf_row0) * fp.width + tx * 32);
#pragma unroll
                    for (int i = 0; i < 3; i++) q[k][i] = __ldcg(reinterpret_cast<const float4*>(rgb + base_v[k] + fill_off[lane + 32 * i]));
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (u0 + k * n_warps < n_units) {               // (uniform over the warp: the shuffles below are converged)
#pragma unroll
                    for (int i = 0; i < 3; i++) {
                        const float4 f = q[k][i];
                        const unsigned w0 = Tone<float>::q(f.x, inv) | (Tone<float>::q(f.y, inv) << 8) | (Tone<float>::q(f.z, inv) << 16) | (Tone<float>::q(f.w, inv) << 24);
                        const unsigned w1 = __shfl_down_sync(0xffffffffu, w0, 1), w2 = __shfl_down_sync(0xffffffffu, w0, 2), w3 = __shfl_down_sync(0xffffffffu, w0, 3);
                        if ((lane & 3) == 0) *reinterpret_cast<uint4*>(rgb8_out + base_v[k] + fill_off[lane + 32 * i]) = make_uint4(w0, w1, w2, w3);
                    }
                }
            }
        }
    }
    // ---- rank 0 of a multi-GPU frame, while the other ranks' tiles are still arriving: the bands of the other ranks are
    // black wherever those ranks store nothing (they only send their busy tiles), so somebody has to clear them -- here,
    // from local HBM bandwidth instead of zeros over NVLink, and for the NEXT frame's buffer (frames alternate between two
    // buffers), in the microseconds this GPU would otherwise spend waiting for the last rank's signal.  The next frame's
    // peers store into that buffer only after this rank has published its next maximum, i.e. after this kernel.
    // A band is 32 full rows = 96 W contiguous bytes; 512-byte pieces are dealt to the grid's warps.
    if (zero_foreign) {
        const int S = fp.row_step >> 5, f = (fp.row_begin >> 5) % S, P = fp.height >> 5;
        const int per_band = fp.width * 96 / 512;                  // W is a multiple of 32: 6 W / 32 pieces
        const int n_foreign = P - (P - f + S - 1) / S;
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        for (int c = blockIdx.x * (kFastBlock / 32) + warp; c < n_foreign * per_band; c += n_warps) {
            const int fb = c / per_band, piece = c - fb * per_band;
            const int g = fb / (S - 1), r = fb - g * (S - 1);
            const int band = g * S + (r < f ? r : r + 1);
            __stcs(reinterpret_cast<uint4*>(rgb8_next + ((size_t)band * fp.width * 96 + (size_t)piece * 512)) + lane, z);
        }
    }
    signal_frame_done(link, ctr + 10);
}

// 16 consecutive channel values per thread -> one 16-byte store.  Rows are W*3 values with W a
// multiple of 32, so every thread's span is 16-byte aligned on both sides.  `band16` = 16-value chunks
// of one 32-row band, `step16` = chunks from the start of one rendered band to the start of the next.
// kPeer: the maximum comes from the ranks' mailboxes and the end of the kernel is signalled (PeerLink).
template <typename R, bool kPeer>
__global__ void __launch_bounds__(256)
tonemap_kernel(const R* __restrict__ rgb, const R* __restrict__ dmax, const int normalise, const size_t first16,
               const size_t count16, const unsigned band16, const size_t step16, unsigned char* __restrict__ rgb8,
               const PeerLink link, int* __restrict__ done) {
    __shared__ float peer_max;
    const size_t l = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    R inv = R(1);
    if (normalise) {
        const R mx = kPeer ? R(gather_max(link, &peer_max)) : *dmax;
        if (mx > R(0)) inv = R(1) / mx;                         // framebuffer.rs:71-76: scale(1. / max_val)
    }
    if (l < count16) {
        const size_t band = l / band16;
        const size_t i = first16 + band * step16 + (l - band * band16);
        const R* src = rgb + i * 16;
        unsigned w[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            R v0, v1, v2, v3;
            if (sizeof(R) == 4) {
                const float4 f = __ldcs(reinterpret_cast<const float4*>(src) + k);
                v0 = f.x; v1 = f.y; v2 = f.z; v3 = f.w;
            } else {
                const double2 a = __ldcs(reinterpret_cast<const double2*>(src) + 2 * k);
                const double2 b = __ldcs(reinterpret_cast<const double2*>(src) + 2 * k + 1);
                v0 = a.x; v1 = a.y; v2 = b.x; v3 = b.y;
            }
            w[k] = Tone<R>::q(v0, inv) | (Tone<R>::q(v1, inv) << 8) | (Tone<R>::q(v2, inv) << 16) | (Tone<R>::q(v3, inv) << 24);
        }
        reinterpret_cast<uint4*>(rgb8)[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (kPeer) signal_frame_done(link, done);
}

// K4 for frames rendered with a tile schedule and rgb8 zero-fill (host API rm_render with out_rgb8, rm_tonemap_device_busy;
// on the frame path this work is the last phase of the render kernel): only the busy tiles (ctr[8] fully covered ones in
// `order`, ctr[9] partially covered ones in `order2`) hold anything but zeros.  A block walks tiles; a thread converts
// one float4 (4 channel values -> 4 bytes) at a time, lanes along a pixel row: 384-byte runs in, 96-byte runs out.
__global__ void __launch_bounds__(256)
tonemap_busy_kernel(const float* __restrict__ rgb, const float* __restrict__ dmax, const int normalise, const FrameParams<float> fp,
                    const int tiles_x, const int* __restrict__ order, const int* __restrict__ order2, const int* __restrict__ ctr,
                    unsigned char* __restrict__ rgb8) {
    const int n_full = ctr[8], n_busy = n_full + ctr[9];
    float inv = 1.f;
    if (normalise) {
        const float mx = *dmax;
        if (mx > 0.f) inv = 1.f / mx;                           // framebuffer.rs:71-76: scale(1. / max_val)
    }
    for (int t = blockIdx.x; t < n_busy; t += gridDim.x) {
        const int tile = t < n_full ? order[t] : order2[t - n_full];
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        const size_t p0 = (size_t)(fp.row_begin + ty * fp.row_step - fp.buf_row0) * fp.width + tx * 32;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const int c = threadIdx.x + 256 * i;                // 768 float4 per tile: 32 rows x 24
            const int row = c / 24, col = c - row * 24;
            const size_t v = 3 * (p0 + (size_t)row * fp.width) + 4 * col;
            const float4 f = __ldcs(reinterpret_cast<const float4*>(rgb + v));
            const unsigned w = Tone<float>::q(f.x, inv) | (Tone<float>::q(f.y, inv) << 8) | (Tone<float>::q(f.z, inv) << 16) | (Tone<float>::q(f.w, inv) << 24);
            *reinterpret_cast<unsigned*>(rgb8 + v) = w;
        }
    }
}

// Host delivery of a tile-scheduled frame (rm_render / rm_render_rows_*), two small kernels after K1.
// (1) The schedule lists the busy tiles in the order K0's atomics happened to hand out; the host wants them in frame order
// (tile index = band * tiles_x + column), so that tiles it scatters one after the other are neighbours in the caller's
// frame.  One CTA: bitmap of the busy tiles in shared memory, prefix sum of the words' popcounts, every word writes its
// tiles at its offset.  sorted[0] = number of busy tiles, sorted[1 + k] = k-th busy tile in frame order.
constexpr int kSortMaxWords = 1024;                             // 32768 tiles: the classify kernel's own limit
__global__ void __launch_bounds__(1024)
sort_busy_kernel(const int* __restrict__ order, const int* __restrict__ order2, const int* __restrict__ ctr, int* __restrict__ sorted) {
    __shared__ unsigned bm[kSortMaxWords];
    __shared__ int off[kSortMaxWords];
    __shared__ int warp_sum[32];
    const int n_full = ctr[8], n_busy = n_full + ctr[9], tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    bm[tid] = 0u;
    __syncthreads();
    for (int t = tid; t < n_busy; t += 1024) {
        const int tile = t < n_full ? order[t] : order2[t - n_full];
        RM_CHECK(tile >= 0 && tile < kSortMaxWords * 32);
        atomicOr(&bm[tile >> 5], 1u << (tile & 31));
    }
    __syncthreads();
    const int c = __popc(bm[tid]);
    int inc = c;                                                // inclusive scan over the 1024 words
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += v;
    }
    if (lane == 31) warp_sum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = warp_sum[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += v;
        }
        warp_sum[lane] = w;
    }
    __syncthreads();
    off[tid] = inc - c + (warp ? warp_sum[warp - 1] : 0);
    if (tid == 0) sorted[0] = n_busy;
    int k = off[tid];
    for (unsigned bits = bm[tid]; bits; bits &= bits - 1) sorted[1 + k++] = tid * 32 + __ffs(bits) - 1;
}
// (2) The busy tiles packed in that order into a contiguous staging buffer -- tile k at floats [3072 k, 3072 (k + 1)),
// rows of 32 pixels -- so that the device-to-host copies move only what is not black (15 % of the cornell frame) and the
// host can scatter a chunk while the next one is still crossing PCIe.  384-byte runs in, 12 KB contiguous out.
__global__ void __launch_bounds__(256)
pack_busy_kernel(const float* __restrict__ rgb, const FrameParams<float> fp, const int tiles_x, const int* __restrict__ sorted,
                 float* __restrict__ packed) {
    const int n_busy = sorted[0];
    for (int t = blockIdx.x; t < n_busy; t += gridDim.x) {
        const int tile = sorted[1 + t];
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        RM_CHECK(tile >= 0 && ty < fp.n_bands && (t == 0 || sorted[t] < tile));
        const size_t p0 = (size_t)(fp.row_begin + ty * fp.row_step - fp.buf_row0) * fp.width + tx * 32;
        float4* dst = reinterpret_cast<float4*>(packed + (size_t)t * 3072);
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const int c = threadIdx.x + 256 * i;                // 768 float4 per tile: 32 rows x 24
            const int row = c / 24, col = c - row * 24;
            __stcs(dst + c, __ldcs(reinterpret_cast<const float4*>(rgb + 3 * (p0 + (size_t)row * fp.width) + 4 * col)));
        }
    }
}

// (3) ... or, when the caller's float32 frame is pinned host memory the device can address, written straight into it:
// tile k of K0's schedule (unsorted: every tile is written exactly once, the order does not matter) goes row by row --
// 384 contiguous bytes each, 24 lanes x 16 bytes -- over PCIe to its place in the frame.  No staging buffer, no scatter on
// the host, whose memory system is what bounds a fresh frame (DESIGN.md 9): the tiles cross it once instead of three times.
__global__ void __launch_bounds__(256)
deliver_busy_kernel(const float* __restrict__ rgb, const FrameParams<float> fp, const int tiles_x, const int* __restrict__ order,
                    const int* __restrict__ order2, const int n_full, const int n_busy, float* __restrict__ host_frame,
                    const size_t host_row_floats) {
    for (int t = blockIdx.x; t < n_busy; t += gridDim.x) {
        const int tile = t < n_full ? order[t] : order2[t - n_full];
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        RM_CHECK(tile >= 0 && ty < fp.n_bands);
        const int y0 = fp.row_begin + ty * fp.row_step;
        const size_t p0 = (size_t)(y0 - fp.buf_row0) * fp.width + tx * 32;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            const int c = threadIdx.x + 256 * i;                // 768 float4 per tile: 32 rows x 24
            const int row = c / 24, col = c - row * 24;
            const float4 v = __ldcs(reinterpret_cast<const float4*>(rgb + 3 * (p0 + (size_t)row * fp.width) + 4 * col));
            *reinterpret_cast<float4*>(host_frame + (size_t)(y0 + row) * host_row_floats + (size_t)tx * 96 + 4 * col) = v;
        }
    }
}

// Supersampled anti-aliasing (rm_render_supersampled): the S x frame box-filtered down to `rows` W-wide output rows
// (rm::resolve_box), and their channel maximum (FrameBuffer::normalize) into *dmax.  A pure streaming pass: 12 S^2 bytes in,
// 12 out per output pixel.  A warp covers 32 consecutive output pixels of one row, so each sub-row it reads is one contiguous
// run of 32 * 12 S bytes; a lane's share of a sub-row (12 S bytes, at a multiple of 12 S from a 16-byte aligned row start:
// W is a multiple of 32) is read as float4 when S is a multiple of 4, as float2 when S is even.
template <int S>
__global__ void __launch_bounds__(256)
resolve_box_kernel(const float* __restrict__ sub, float* __restrict__ out, const int width, const int rows,
                   float* __restrict__ dmax) {
    __shared__ int cta_max;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) cta_max = 0;
    __syncthreads();
    const int warps_x = width >> 5;
    const long long g = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int y = (int)(g / warps_x);
    const int x = (int)(g - (long long)y * warps_x) * 32 + lane;
    float m = 0.f;
    if (y < rows) {
        const size_t sub_row = (size_t)S * width * 3;          // floats per row of the S x frame
        const float* p = sub + (size_t)S * y * sub_row + (size_t)S * 3 * x;
        float o[3];
        resolve_box<S>([&](int i, float (&r)[3 * S]) {
            const float* q = p + i * sub_row;
            if constexpr (S % 4 == 0) {
#pragma unroll
                for (int k = 0; k < 3 * S / 4; k++) {
                    const float4 f = reinterpret_cast<const float4*>(q)[k];
                    r[4 * k] = f.x; r[4 * k + 1] = f.y; r[4 * k + 2] = f.z; r[4 * k + 3] = f.w;
                }
            } else if constexpr (S % 2 == 0) {
#pragma unroll
                for (int k = 0; k < 3 * S / 2; k++) {
                    const float2 f = reinterpret_cast<const float2*>(q)[k];
                    r[2 * k] = f.x; r[2 * k + 1] = f.y;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 3 * S; k++) r[k] = q[k];
            }
        }, o);
        float* d = out + ((size_t)y * width + x) * 3;
        d[0] = o[0]; d[1] = o[1]; d[2] = o[2];
        m = fmaxf(fmaxf(o[0], o[1]), o[2]);
    }
    // values are >= 0, so the integer order of the bit patterns is the float order
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomicMax(&cta_max, wm);
    __syncthreads();
    if (threadIdx.x == 0 && cta_max > 0) atomicMax(reinterpret_cast<int*>(dmax), cta_max);
}

// ---- Adaptive anti-aliasing (rm_render_adaptive): mark -> sub-pixel rays of the marked pixels -> resolve ----------------
// Mark: one thread per pixel of the call's n_px = rows * W pixels from frame row row_begin (a warp: 32 pixels of one row,
// W being a multiple of 32).  The 1x frame (rgb, id) holds rows [lo, hi).  Pixels that are not refined keep their 1x value,
// which is already in place in rgb, and fold it into *dmax; refined ones go to `list` as x | y << 16 (one atomic per warp:
// the order of the list varies from run to run, what is computed for each entry does not).  mask[i]: 1 = refined.
__global__ void __launch_bounds__(256)
adaptive_mark_kernel(const float* __restrict__ rgb, const int* __restrict__ id, const int width, const int lo, const int hi,
                     const int row_begin, const long long n_px, const float k, const int all, unsigned char* __restrict__ mask,
                     unsigned* __restrict__ list, unsigned* __restrict__ count, float* __restrict__ dmax) {
    __shared__ int cta_max;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) cta_max = 0;
    __syncthreads();
    const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
    bool refine = false;
    float m = 0.f;
    int x = 0, y = 0;
    if (t < n_px) {
        const long long r = t / width;
        y = row_begin + (int)r;
        x = (int)(t - r * width);
        refine = adaptive_mark(rgb, id, width, lo, hi, x, y, k, all != 0);
        mask[t] = refine ? 1 : 0;
        if (!refine) {
            const float* v = rgb + 3 * ((size_t)(y - lo) * width + x);
            m = fmaxf(fmaxf(v[0], v[1]), v[2]);
        }
    }
    const unsigned b = __ballot_sync(0xffffffffu, refine);
    if (b) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(count, (unsigned)__popc(b));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (refine) list[base + __popc(b & ((1u << lane) - 1u))] = (unsigned)x | ((unsigned)y << 16);
    }
    // values are >= 0, so the integer order of the bit patterns is the float order
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomicMax(&cta_max, wm);
    __syncthreads();
    if (threadIdx.x == 0 && cta_max > 0) atomicMax(reinterpret_cast<int*>(dmax), cta_max);
}

// Sub-pixel rays of the listed pixels: entry e of the list, sub-pixel r = i * s + j (i, j in [0, s)), is the s x frame's
// pixel (s x + j, s y + i), and its value goes to sub[3 (e s^2 + r) ...] -- every listed pixel's s^2 values contiguous,
// sub-rows outer, in resolve_box's order.  fp is the s x frame's FrameParams.  Every value is the one render_fast_kernel
// (K1) writes for that pixel of the s x frame, bit for bit: the same device functions with the same operands per pixel --
// primary_begin, primary_tri over the raster records K0 wrote for this camera (they depend on the camera only, not on the
// frame size) or primary_bvh, primary_rest, fast_shade -- and misses are 0.
// Persistent grid: a warp draws 32 consecutive sub-rays at a time from a 64-bit counter (*next, zero at launch) up to
// *count * s^2 -- the list length stays on the device.  Stage A runs one sub-ray per lane; the warp's triangles are first
// bounded against the rectangle of its 32 sub-pixels (tri_may_touch: exact, see rect_max).  Hits go to the warp's queue,
// compacted with ballot / popc, and are shaded 32 at a time (stage B on full warps, like K1); the last partial round runs
// when the work has run out.
constexpr int kAdaptiveQueue = 64;
template <bool kSmem, bool kBvh, int kGlass>
__global__ void __launch_bounds__(kFastBlock, RM_K1_MIN_BLOCKS)
adaptive_subpixel_kernel(const DeviceScene<float> ds, const FrameParams<float> fp, const int cull, const int samples,
                         const unsigned* __restrict__ list, const unsigned* __restrict__ count,
                         unsigned long long* __restrict__ next, float* __restrict__ sub, const int stage_mat) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    __shared__ float4 queue[kFastBlock / 32][kAdaptiveQueue];       // {t, slot, id, sub-ray index}
    const BlobLayout& L = ds.lay;
    const int n_tri = tri_count(L, cull != 0);
    const unsigned char* base = ds.blob;
    const R4<float>* tri_r = ds.tri_r;
    if (kSmem) {                                                // as K1: blob | raster records | materials (if they fit)
        const uint4* src = reinterpret_cast<const uint4*>(ds.blob);
        uint4* dst = reinterpret_cast<uint4*>(smem_raw);
        const int n16 = L.bytes / 16;
        for (int i = threadIdx.x; i < n16; i += kFastBlock) dst[i] = __ldg(src + i);
        const uint4* rsrc = reinterpret_cast<const uint4*>(ds.tri_r);
        for (int i = threadIdx.x; i < n_tri * 4; i += kFastBlock) dst[n16 + i] = rsrc[i];
        if (stage_mat) {
            uint4* m = dst + n16 + L.n_tri * 4;
            const uint4* a = reinterpret_cast<const uint4*>(ds.mat_a);
            const uint4* b = reinterpret_cast<const uint4*>(ds.mat_b);
            for (int i = threadIdx.x; i < ds.n_mat; i += kFastBlock) {
                m[i] = __ldg(a + i);
                m[ds.n_mat + i] = __ldg(b + i);
                reinterpret_cast<int*>(m + 2 * ds.n_mat)[i] = __ldg(ds.mat_f + i);
            }
        }
        base = smem_raw;
        tri_r = reinterpret_cast<const R4<float>*>(smem_raw + L.bytes);
    }
    __syncthreads();
    FastViewT<kBvh, false> fv;
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
    if (kSmem && stage_mat) {
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

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lane_lt = (1u << lane) - 1u;
    const bool rest = fv.n_sph + fv.n_poly > 0;
    const unsigned ss = (unsigned)(samples * samples);
    const unsigned long long total = (unsigned long long)*count * ss;
    float4* const wq = queue[warp];
    int qn = 0;                                                 // entries in this warp's queue (warp-uniform)
    // sub-ray g -> its pixel of the s x frame
    auto sub_pixel = [&](const unsigned long long g, int& sx, int& sy) {
        const unsigned long long e = g / ss;
        const int r = (int)(g - e * ss), i = r / samples, j = r - i * samples;
        const unsigned xy = __ldg(list + e);
        sx = samples * (int)(xy & 0xffffu) + j;
        sy = samples * (int)(xy >> 16) + i;
    };
    auto shade_entry = [&](const float4 e) {
        const unsigned long long g = (unsigned long long)__float_as_uint(e.w);
        int sx, sy;
        sub_pixel(g, sx, sy);
        RM_CHECK(g < total && sx >= 0 && sx < fp.width && sy >= 0 && sy < fp.height);
        const Vec3<float> c = fast_shade<kGlass>(fv, fp, sx, sy, e.x, __float_as_int(e.y), __float_as_int(e.z));
        float* dst = sub + 3 * g;
        dst[0] = c.x;
        dst[1] = c.y;
        dst[2] = c.z;
    };
    for (;;) {
        unsigned long long g0 = 0;
        if (lane == 0) g0 = atomicAdd(next, 32ull);
        g0 = __shfl_sync(0xffffffffu, g0, 0);
        if (g0 >= total) break;
        const unsigned long long g = g0 + lane;
        const bool live = g < total;
        int sx = 0, sy = 0;
        if (live) sub_pixel(g, sx, sy);
        PrimaryState<1> ps;
        primary_begin<1>(ps, fp, sx, sy);
        if constexpr (kBvh) {
            primary_bvh<1, false>(ps, fv, fp);
        } else {
            // the rectangle of the warp's live sub-pixels (lane 0 is always live)
            const int xa = __reduce_min_sync(0xffffffffu, live ? sx : 0x7fffffff), xb = __reduce_max_sync(0xffffffffu, live ? sx : -1);
            const int ya = __reduce_min_sync(0xffffffffu, live ? sy : 0x7fffffff), yb = __reduce_max_sync(0xffffffffu, live ? sy : -1);
            const float Xa = pixel_X(fp, xa), Xb = pixel_X(fp, xb), Ya = pixel_Y(fp, ya), Yb = pixel_Y(fp, yb);
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
        const bool hit = live && ps.slot[0] >= 0;
        if (live && !hit) {                                     // renderer.rs:300-306: a primary miss is black
            float* dst = sub + 3 * g;
            dst[0] = 0.f;
            dst[1] = 0.f;
            dst[2] = 0.f;
        }
        const unsigned mh = __ballot_sync(0xffffffffu, hit);
        RM_CHECK(qn + __popc(mh) <= kAdaptiveQueue);
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
}

// Resolve of the refined pixels: list entry e's s^2 sub-pixel values (sub, laid out as above) -> rm::resolve_box<S> -> its
// pixel of rgb (rows from frame row lo), and their maximum into *dmax.  Grid-stride over the *count entries.
template <int S>
__global__ void __launch_bounds__(256)
adaptive_resolve_kernel(const float* __restrict__ sub, const unsigned* __restrict__ list, const unsigned* __restrict__ count,
                        float* __restrict__ rgb, const int width, const int lo, float* __restrict__ dmax) {
    __shared__ int cta_max;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) cta_max = 0;
    __syncthreads();
    const unsigned n = *count;
    float m = 0.f;
    for (unsigned e = blockIdx.x * 256u + threadIdx.x; e < n; e += gridDim.x * 256u) {
        const unsigned xy = list[e];
        const int x = (int)(xy & 0xffffu), y = (int)(xy >> 16);
        const float* p = sub + (size_t)e * (3 * S * S);
        float o[3];
        resolve_box<S>([&](int i, float (&r)[3 * S]) {
#pragma unroll
            for (int k = 0; k < 3 * S; k++) r[k] = p[i * 3 * S + k];
        }, o);
        float* d = rgb + 3 * ((size_t)(y - lo) * width + x);
        d[0] = o[0]; d[1] = o[1]; d[2] = o[2];
        m = fmaxf(m, fmaxf(fmaxf(o[0], o[1]), o[2]));
    }
    const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(m));
    if (lane == 0 && wm > 0) atomicMax(&cta_max, wm);
    __syncthreads();
    if (threadIdx.x == 0 && cta_max > 0) atomicMax(reinterpret_cast<int*>(dmax), cta_max);
}

__global__ void publish_zero_kernel(const PeerLink link, float* __restrict__ dmax) {
    *dmax = 0.f;
    publish_max(link, 0.f);
}

__global__ void __launch_bounds__(256) ffma_probe_kernel(float* __restrict__ sink, const int iters) {
    const float b = 0.9999999f, c = 1e-7f;
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = (float)(threadIdx.x + k) * 1e-3f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = fmaf(a[k], b, c);
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = fmaf(a[k], b, c);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace

namespace {
cudaError_t launch_fast(const DeviceScene<float>& ds, const FrameParams<float>& fp, bool cull, float* rgb, int* prim_id,
                        float* dmax, cudaStream_t stream, const double camera[3], int* launches, RenderExtras* ex) {
    unsigned char* rgb8 = ex ? ex->rgb8_zero : nullptr;
    if (ex && ex->ev_begin) cudaEventRecord(ex->ev_begin, stream);
    const int n_tri = tri_count(ds.lay, cull);
    const int tiles_x = fp.width / kFastTile, n_tiles = tiles_x * fp.n_bands;
    const bool bvh = fp.accel != 0 && ds.bvh.n_nodes > 0 && ds.lay.n_lgt <= kBvhMaxLights;
    const bool classify = !bvh && ds.lay.n_sph + poly_count(ds.lay, cull) == 0 && n_tri <= kClassifyMaxTris && n_tiles <= ds.tile_order_cap / 2;
    if (classify)
        prepare_classify_kernel<<<(n_tiles * kClassifyLanes + kClassifyBlock - 1) / kClassifyBlock, kClassifyBlock, 0, stream>>>(ds.tri_src, n_tri, camera[0], camera[1], camera[2], ds.tri_r,
                                                                         fp, tiles_x, n_tiles, ds.tile_order, ds.tile_order + ds.tile_order_cap / 2, ds.ctr,
                                                                         ex && ex->zero_dmax ? dmax : nullptr);
    else
        prepare_raster_kernel<<<(std::max(n_tri, 1) + 127) / 128, 128, 0, stream>>>(ds.tri_src, n_tri, camera[0], camera[1], camera[2], ds.tri_r,
                                                                                     ex && ex->zero_dmax ? dmax : nullptr);
    const PeerLink link = ex ? ex->link : PeerLink();
    const int* order = classify ? ds.tile_order : nullptr;
    if (ex) ex->scheduled = classify;
    if (!classify) rgb8 = nullptr;                              // without a schedule the tone-map kernel converts every tile
    unsigned char* rgb8_out = ex ? ex->rgb8_out : nullptr;     // fused K4 (needs a link: the mailbox wait is its barrier)
    if (link.world <= 0) rgb8_out = nullptr;
    const int normalise = ex && ex->normalise ? 1 : 0;
    // rank 0 of a multi-GPU frame clears the other ranks' bands of the NEXT frame's buffer at the end of this kernel
    unsigned char* rgb8_next = (rgb8_out && link.world > 1 && link.rank == 0) ? ex->rgb8_next : nullptr;
    if (ex && ex->ev_prepared) cudaEventRecord(ex->ev_prepared, stream);      // (an event here gives up the overlap of K1's launch with K0)
    if (launches) (*launches)++;
    // shared memory: scene blob | raster records of every fast-path triangle | materials (if they fit as well), next to the
    // kernel's static arrays (hit queues etc.) within the opt-in limit of the device
    static int sm_count = 0, dyn_limit = 0;
    cudaError_t e;
    if (!sm_count) {
        int dev = 0, optin = 0;
        cudaFuncAttributes fa;
        if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
        if ((e = cudaFuncGetAttributes(&fa, render_fast_kernel<true, 0, GLASS_F64>)) != cudaSuccess) return e;
        dyn_limit = std::min(kSmemLimit, optin - (int)fa.sharedSizeBytes - 1024);
        if ((e = cudaFuncSetAttribute(render_fast_kernel<true, 0, GLASS_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(render_fast_kernel<true, 0, GLASS_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit)) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(render_fast_kernel<true, 0, GLASS_F64>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    }
    const size_t smem_geo = (size_t)ds.lay.bytes + (size_t)ds.lay.n_tri * 64;
    const size_t smem_mat = (((size_t)ds.n_mat * 36) + 15) / 16 * 16;
    const int stage_mat = smem_geo + smem_mat <= (size_t)dyn_limit ? 1 : 0;
    const size_t smem = smem_geo + (stage_mat ? smem_mat : 0);
    const float inv_tiles_x = 1.0f / (float)tiles_x;
    // launched with programmatic stream serialisation: the CTAs may become resident while K0 still runs (pdl_wait_primary)
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kFastBlock);
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // The fused exchange + K4 phase waits inside the kernel for a word that is published only when EVERY CTA of the grid
    // has retired from rendering: all CTAs must be resident together.  The grid is sized from the occupancy API, which
    // makes that true on a GPU this process has to itself (include/rm_b200.h, rm_render_frame: "sharing the device");
    // a cooperative launch makes the driver guarantee it whatever else runs on the device, at the price of the launch
    // overlap with K0 (measured: +2 to 3 us on a 70 us frame).  RM_B200_COOPERATIVE=1 asks for it; a driver that refuses
    // the attribute together with the programmatic launch edge switches it off again for the process.
    static int coop = -1;
    if (coop < 0) {
        const char* env = getenv("RM_B200_COOPERATIVE");
        coop = (env && env[0] == '1') ? 1 : 0;
    }
    const bool want_coop = coop == 1 && link.world > 0 && rgb8_out != nullptr;
    if (want_coop) {
        attr[1].id = cudaLaunchAttributeCooperative;
        attr[1].val.cooperative = 1;
        cfg.numAttrs = 2;
    }
    const int cull_i = cull ? 1 : 0;
    const int* order2 = order ? ds.tile_order + ds.tile_order_cap / 2 : nullptr;
    const bool use_smem = !bvh && smem <= (size_t)dyn_limit;
    // the reflect / refract recursion only where a frame can need it, its f64 ray geometry only where FP32 would not do
    const int glass = glass_mode(ds.lay.any_glass != 0, ds.lay.n_sph, ds.lay.coord_max, ds.lay.r_min, camera);
    if (ex) ex->glass_mode = glass;
    using K1 = decltype(&render_fast_kernel<true, 0, GLASS_NONE>);
    static const K1 table[4][3] = {
        {render_fast_kernel<true, 0, GLASS_NONE>, render_fast_kernel<true, 0, GLASS_F32>, render_fast_kernel<true, 0, GLASS_F64>},
        {render_fast_kernel<false, 0, GLASS_NONE>, render_fast_kernel<false, 0, GLASS_F32>, render_fast_kernel<false, 0, GLASS_F64>},
        {render_fast_kernel<false, 1, GLASS_NONE>, render_fast_kernel<false, 1, GLASS_F32>, render_fast_kernel<false, 1, GLASS_F64>},
        {render_fast_kernel<false, 2, GLASS_NONE>, render_fast_kernel<false, 2, GLASS_F32>, render_fast_kernel<false, 2, GLASS_F64>}};
    const K1 k = table[bvh ? (fp.accel == 2 ? 3 : 2) : use_smem ? 0 : 1][glass];
    cfg.dynamicSmemBytes = use_smem ? smem : 0;
    int occ = 1;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kFastBlock, cfg.dynamicSmemBytes)) != cudaSuccess) return e;
    cfg.gridDim = dim3(std::min(n_tiles, sm_count * std::max(occ, 1)));
    e = cudaLaunchKernelEx(&cfg, k, ds, fp, cull_i, tiles_x, n_tiles, inv_tiles_x, rgb, prim_id, dmax, ds.ctr, order, order2, rgb8,
                           link, rgb8_out, normalise, rgb8_next, stage_mat);
    if (e != cudaSuccess && want_coop) {                        // not available in this combination: the plain persistent launch
        cudaGetLastError();
        coop = 0;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, k, ds, fp, cull_i, tiles_x, n_tiles, inv_tiles_x, rgb, prim_id, dmax, ds.ctr, order, order2, rgb8,
                               link, rgb8_out, normalise, rgb8_next, stage_mat);
    }
    if (e != cudaSuccess) return e;
    if (launches) (*launches)++;
    if (ex && ex->ev_rendered) cudaEventRecord(ex->ev_rendered, stream);
    return cudaGetLastError();
}
cudaError_t launch_fast(const DeviceScene<double>&, const FrameParams<double>&, bool, double*, int*, double*, cudaStream_t,
                        const double*, int*, RenderExtras*) { return cudaErrorInvalidValue; }
}  // namespace

template <typename R>
cudaError_t launch_render(const DeviceScene<R>& ds, const FrameParams<R>& fp, bool cull, R* rgb, int* prim_id, R* dmax,
                          unsigned long long* counters, cudaStream_t stream, const double camera[3], int* launches,
                          RenderExtras* ex) {
    const int rows = fp.n_bands * 32;
    if (ex) ex->scheduled = false;
    if (rows <= 0 || fp.width <= 0) {                           // nothing to render: the profiling events still mark the (empty) frame
        if (ex && ex->ev_begin) cudaEventRecord(ex->ev_begin, stream);
        if (ex && ex->ev_prepared) cudaEventRecord(ex->ev_prepared, stream);
        if (ex && ex->ev_rendered) cudaEventRecord(ex->ev_rendered, stream);
        return cudaSuccess;
    }
    const dim3 grid((fp.width + kTileW - 1) / kTileW, (rows + kTileH - 1) / kTileH);
    // (a depth cap of 0 makes every pixel the background, hit or not -- renderer.rs:262-264 with n_recursion = 1: the generic
    // kernel follows cast_ray literally, the production kernel assumes at least the primary level)
    if (sizeof(R) == 4 && !counters && camera && ds.tri_r && fp.max_depth >= 1) return launch_fast(ds, fp, cull, rgb, prim_id, dmax, stream, camera, launches, ex);
    if (ex && ex->ev_begin) cudaEventRecord(ex->ev_begin, stream);
    if (ex && ex->ev_prepared) cudaEventRecord(ex->ev_prepared, stream);
    if (launches) (*launches)++;
    const int use_smem = ds.lay.bytes <= kSmemLimit;
    const size_t smem = use_smem ? (size_t)ds.lay.bytes : 0;
    cudaError_t e;
    if (counters) {
        auto k = render_kernel<R, true>;
        if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        k<<<grid, kBlock, smem, stream>>>(ds, fp, cull ? 1 : 0, use_smem, rgb, prim_id, dmax, counters);
    } else {
        auto k = render_kernel<R, false>;
        if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        k<<<grid, kBlock, smem, stream>>>(ds, fp, cull ? 1 : 0, use_smem, rgb, prim_id, dmax, nullptr);
    }
    if (ex && ex->ev_rendered) cudaEventRecord(ex->ev_rendered, stream);
    return cudaGetLastError();
}

cudaError_t launch_tonemap_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, const float* dmax,
                                bool normalise, unsigned char* rgb8, cudaStream_t stream) {
    const int tiles_x = fp.width / kFastTile, n_tiles = tiles_x * fp.n_bands;
    if (n_tiles <= 0) return cudaSuccess;
    const int blocks = std::min(n_tiles, 148 * 8);
    tonemap_busy_kernel<<<blocks, 256, 0, stream>>>(rgb, dmax, normalise ? 1 : 0, fp, tiles_x, ds.tile_order,
                                                    ds.tile_order + ds.tile_order_cap / 2, ds.ctr, rgb8);
    return cudaGetLastError();
}

cudaError_t launch_pack_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, int* sorted, float* packed,
                             cudaStream_t stream) {
    const int tiles_x = fp.width / kFastTile, n_tiles = tiles_x * fp.n_bands;
    if (n_tiles <= 0) return cudaSuccess;
    if (n_tiles > kSortMaxWords * 32) return cudaErrorInvalidValue;
    sort_busy_kernel<<<1, 1024, 0, stream>>>(ds.tile_order, ds.tile_order + ds.tile_order_cap / 2, ds.ctr, sorted);
    pack_busy_kernel<<<std::min(n_tiles, 148 * 8), 256, 0, stream>>>(rgb, fp, tiles_x, sorted, packed);
    return cudaGetLastError();
}

cudaError_t launch_deliver_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, int n_full, int n_busy,
                                float* host_frame, size_t host_row_floats, cudaStream_t stream) {
    const int tiles_x = fp.width / kFastTile;
    if (n_busy <= 0) return cudaSuccess;
    deliver_busy_kernel<<<std::min(n_busy, 148 * 8), 256, 0, stream>>>(rgb, fp, tiles_x, ds.tile_order, ds.tile_order + ds.tile_order_cap / 2,
                                                                       n_full, n_busy, host_frame, host_row_floats);
    return cudaGetLastError();
}

cudaError_t launch_resolve_box(const float* sub, int samples, float* out, int width, int rows, float* dmax, cudaStream_t stream) {
    const long long warps = (long long)(width / 32) * rows;
    if (warps <= 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((warps + 7) / 8);
    switch (samples) {
        case 1: resolve_box_kernel<1><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 2: resolve_box_kernel<2><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 3: resolve_box_kernel<3><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 4: resolve_box_kernel<4><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 5: resolve_box_kernel<5><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 6: resolve_box_kernel<6><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 7: resolve_box_kernel<7><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        case 8: resolve_box_kernel<8><<<blocks, 256, 0, stream>>>(sub, out, width, rows, dmax); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_adaptive_mark(const float* rgb, const int* id, int width, int lo, int hi, int row_begin, int rows, float k,
                                 bool all, unsigned char* mask, unsigned* list, unsigned* count, float* dmax, cudaStream_t stream) {
    const long long n_px = (long long)width * rows;
    if (n_px <= 0) return cudaSuccess;
    adaptive_mark_kernel<<<(unsigned)((n_px + 255) / 256), 256, 0, stream>>>(rgb, id, width, lo, hi, row_begin, n_px, k, all ? 1 : 0,
                                                                             mask, list, count, dmax);
    return cudaGetLastError();
}

cudaError_t launch_adaptive_subpixel(const DeviceScene<float>& ds, const FrameParams<float>& fp, bool cull, int samples,
                                     const unsigned* list, const unsigned* count, unsigned long long* next, float* sub,
                                     const double camera[3], cudaStream_t stream) {
    // the instantiation launch_fast would pick for this scene and camera: hierarchy or not, glass mode, staged scene
    using K = decltype(&adaptive_subpixel_kernel<true, false, GLASS_NONE>);
    static const K table[3][3] = {
        {adaptive_subpixel_kernel<true, false, GLASS_NONE>, adaptive_subpixel_kernel<true, false, GLASS_F32>, adaptive_subpixel_kernel<true, false, GLASS_F64>},
        {adaptive_subpixel_kernel<false, false, GLASS_NONE>, adaptive_subpixel_kernel<false, false, GLASS_F32>, adaptive_subpixel_kernel<false, false, GLASS_F64>},
        {adaptive_subpixel_kernel<false, true, GLASS_NONE>, adaptive_subpixel_kernel<false, true, GLASS_F32>, adaptive_subpixel_kernel<false, true, GLASS_F64>}};
    static int sm_count = 0, dyn_limit = 0;
    cudaError_t e;
    if (!sm_count) {
        int dev = 0, optin = 0;
        cudaFuncAttributes fa;
        if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
        if ((e = cudaFuncGetAttributes(&fa, table[0][GLASS_F64])) != cudaSuccess) return e;
        dyn_limit = std::min(kSmemLimit, optin - (int)fa.sharedSizeBytes - 1024);
        for (int gm = 0; gm < 3; gm++)
            if ((e = cudaFuncSetAttribute(table[0][gm], cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_limit)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    }
    const bool bvh = fp.accel != 0 && ds.bvh.n_nodes > 0 && ds.lay.n_lgt <= kBvhMaxLights;
    const size_t smem_geo = (size_t)ds.lay.bytes + (size_t)ds.lay.n_tri * 64;
    const size_t smem_mat = (((size_t)ds.n_mat * 36) + 15) / 16 * 16;
    const int stage_mat = smem_geo + smem_mat <= (size_t)dyn_limit ? 1 : 0;
    const size_t smem = smem_geo + (stage_mat ? smem_mat : 0);
    const bool use_smem = !bvh && smem <= (size_t)dyn_limit;
    const int glass = glass_mode(ds.lay.any_glass != 0, ds.lay.n_sph, ds.lay.coord_max, ds.lay.r_min, camera);
    const K k = table[bvh ? 2 : use_smem ? 0 : 1][glass];
    const size_t dyn = use_smem ? smem : 0;
    int occ = 1;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kFastBlock, dyn)) != cudaSuccess) return e;
    k<<<sm_count * std::max(occ, 1), kFastBlock, dyn, stream>>>(ds, fp, cull ? 1 : 0, samples, list, count, next, sub, stage_mat);
    return cudaGetLastError();
}

cudaError_t launch_adaptive_resolve(const float* sub, int samples, const unsigned* list, const unsigned* count, float* rgb, int width,
                                    int lo, long long max_entries, float* dmax, cudaStream_t stream) {
    if (max_entries <= 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<long long>((max_entries + 255) / 256, 148 * 8);
    switch (samples) {
        case 1: adaptive_resolve_kernel<1><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 2: adaptive_resolve_kernel<2><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 3: adaptive_resolve_kernel<3><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 4: adaptive_resolve_kernel<4><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 5: adaptive_resolve_kernel<5><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 6: adaptive_resolve_kernel<6><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 7: adaptive_resolve_kernel<7><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        case 8: adaptive_resolve_kernel<8><<<blocks, 256, 0, stream>>>(sub, list, count, rgb, width, lo, dmax); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

namespace {
template <typename R, bool kPeer>
cudaError_t launch_tonemap_impl(const FrameParams<R>& fp, const R* rgb, const R* dmax, bool normalise, unsigned char* rgb8,
                                cudaStream_t stream, const PeerLink& link, int* done) {
    const int rows = fp.n_bands * 32;
    if (rows <= 0 && !kPeer) return cudaSuccess;
    // both buffers are indexed from pixel row fp.buf_row0
    const size_t row16 = (size_t)fp.width * 3 / 16;
    const size_t first16 = (size_t)(fp.row_begin - fp.buf_row0) * row16;
    const size_t count16 = (size_t)std::max(rows, 0) * row16;
    const int blocks = std::max((int)((count16 + 255) / 256), 1);
    tonemap_kernel<R, kPeer><<<blocks, 256, 0, stream>>>(rgb, dmax, normalise ? 1 : 0, first16, count16, (unsigned)std::max<size_t>(32 * row16, 1),
                                                         (size_t)fp.row_step * row16, rgb8, link, done);
    return cudaGetLastError();
}
}  // namespace

template <typename R>
cudaError_t launch_tonemap(const FrameParams<R>& fp, const R* rgb, const R* dmax, bool normalise, unsigned char* rgb8,
                           cudaStream_t stream) {
    return launch_tonemap_impl<R, false>(fp, rgb, dmax, normalise, rgb8, stream, PeerLink(), nullptr);
}

cudaError_t launch_tonemap_peer(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, const float* dmax,
                                bool normalise, unsigned char* rgb8, cudaStream_t stream, const PeerLink& link) {
    return launch_tonemap_impl<float, true>(fp, rgb, dmax, normalise, rgb8, stream, link, ds.ctr + 10);
}

cudaError_t launch_publish_zero(const PeerLink& link, float* dmax, cudaStream_t stream) {
    publish_zero_kernel<<<1, 1, 0, stream>>>(link, dmax);
    return cudaGetLastError();
}

cudaError_t launch_ffma_probe(float* sink, int iters, int blocks, cudaStream_t stream, double* flops) {
    ffma_probe_kernel<<<blocks, 256, 0, stream>>>(sink, iters);
    if (flops) *flops = (double)blocks * 256.0 * (double)iters * 16.0 * 2.0;
    return cudaGetLastError();
}

template cudaError_t launch_render<float>(const DeviceScene<float>&, const FrameParams<float>&, bool, float*, int*, float*, unsigned long long*, cudaStream_t, const double*, int*, RenderExtras*);
template cudaError_t launch_render<double>(const DeviceScene<double>&, const FrameParams<double>&, bool, double*, int*, double*, unsigned long long*, cudaStream_t, const double*, int*, RenderExtras*);
template cudaError_t launch_tonemap<float>(const FrameParams<float>&, const float*, const float*, bool, unsigned char*, cudaStream_t);
template cudaError_t launch_tonemap<double>(const FrameParams<double>&, const double*, const double*, bool, unsigned char*, cudaStream_t);

}  // namespace rm
