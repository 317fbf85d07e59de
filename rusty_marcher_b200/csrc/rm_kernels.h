// rm_kernels.h -- launchers of the sm_100a kernels (rm_kernels.cu), used by the C ABI (rm_api.cu).
#pragma once

#include <cuda_runtime.h>

#include "rm_scene.h"

namespace rm {

// The packed scene in HBM (see rm_scene.h for the blob layout).
template <typename R> struct DeviceScene {
    const unsigned char* blob = nullptr;
    BlobLayout lay;
    const R4<R>* mat_a = nullptr;
    const R4<R>* mat_b = nullptr;
    const int* mat_f = nullptr;
    int n_mat = 0;                                   // entries of mat_a / mat_b / mat_f (= primitives of the scene)
    const int* order[2] = {nullptr, nullptr};        // [0] every primitive, [1] after culling
    const int* order_shape[2] = {nullptr, nullptr};
    int n_order[2] = {0, 0};
    // FP32 fast path: FP64 triangle sources (input of the per-frame prepare kernel) and the
    // camera-specialised raster records it writes (4 x R4<float> per triangle, rebuilt every frame)
    const double* tri_src = nullptr;
    R4<float>* tri_r = nullptr;
    // FP32 pack: f64 {c, r^2} per sphere and {n, n.C} per plane slot, read by the f64 ray geometry of glass paths (cast_glass)
    const double* sph64 = nullptr;
    const double* pln64 = nullptr;
    // frame control block of the persistent render kernel, zero between frames (the last CTA to finish resets it):
    //   ctr[0] next busy tile   ctr[1] fully covered tiles   ctr[2] empty tiles   ctr[3] CTAs finished   ctr[5] partially covered tiles
    //   ctr[6..7] u64: scene queries behind the primary rays, accumulated by the hierarchy kernel (rm_scene_query_count)
    int* ctr = nullptr;
    // tile schedule written by the classify kernel: busy tiles (some triangle may touch them) first, then the
    // tiles that are provably empty and only need their black pixels stored
    int* tile_order = nullptr;
    int tile_order_cap = 0;
    // hierarchy over the hittable primitives (rm_bvh.cuh), walked instead of the flat arrays when RmParams.accel is set
    BvhView bvh;
};

// The path's one exchange step (SURVEY.md 8e) done by the kernels themselves over peer memory (NVLink): every rank owns
// a mailbox of kMailboxWords 64-bit words that all ranks of the box have mapped (CUDA IPC).
//   word [(seq & 1) * 16 + src]   {seq, max bits} published by rank src's render kernel (double buffered by frame parity:
//                                 a rank may be at most one frame ahead of the slowest reader, see DESIGN.md)
//   word [32 + src]               {seq, 1} on rank 0 only: rank src's tone-map kernel has stored all its bytes of the frame
//   word [48]                     non-zero when a wait gave up after kPeerTimeoutNs (a peer died); sticky
//   words [56, 61)                %globaltimer stamps (ns) of the rank's last frame: kernel start, rendering done, maxima
//                                 gathered, own bytes stored, (rank 0) frame complete -- rm_peer_stamps()
constexpr int kMaxRanks = 16;
constexpr int kMailboxWords = 64;
struct PeerLink {
    int rank = 0, world = 0;            // world == 0: no exchange (single-GPU calls)
    unsigned seq = 0;                   // frame sequence number, >= 1, the same on every rank
    unsigned long long* box[kMaxRanks] = {};
};

// Optional extras of a render launch.
struct RenderExtras {
    // in: let K0 zero *dmax (saves the memset launch of frame-level calls)
    bool zero_dmax = false;
    // in: publish the channel maximum of this rank's rows to every rank's mailbox when the render kernel retires
    PeerLink link;
    // in: the 8-bit frame (indexed like rgb).  When the frame gets a tile schedule the render kernel zeroes the bytes of
    // every pixel it visits, so that launch_tonemap_busy() only has to convert the busy tiles afterwards.
    unsigned char* rgb8_zero = nullptr;
    // in: fuse K4 into the render kernel (needs `link`): once every rank's maximum is in this rank's mailbox the kernel
    // converts its busy tiles (all its tiles without a schedule) into rgb8_out, which may be peer memory, and signals rank 0
    unsigned char* rgb8_out = nullptr;
    bool normalise = true;
    // in (rank 0 of a multi-GPU frame): the 8-bit buffer of the NEXT frame, whose foreign bands this launch clears
    unsigned char* rgb8_next = nullptr;
    // in: events recorded on the stream before K0, between K0 and K1, after K1 (profiling; may be null)
    cudaEvent_t ev_begin = nullptr, ev_prepared = nullptr, ev_rendered = nullptr;
    // out: the frame was rendered with a tile schedule (and rgb8_zero, if given, has been zero-filled)
    bool scheduled = false;
    // out: GlassMode of the production kernel that was launched (rm_fast.cuh)
    int glass_mode = 0;
};

// K0 + K1.  With counters == null and R = float this is the production path: prepare_raster_kernel
// (one thread per triangle, FP64) followed by render_fast_kernel; otherwise the generic kernel.
// K1: render rows [fp.row_begin, fp.row_end).  rgb: H*W*3 of R; prim_id optional; dmax: scalar R that
// receives max(old, tile max); counters: 17 x u64 (instrumented kernel) or null (production kernel).
// view: the camera's orientation (rm_render_view), or null for the reference's camera looking down -z.  Under a view the
// hierarchy kernel that counts its work (accel = 2) is not instantiated: accel = 2 renders as accel = 1.
template <typename R>
cudaError_t launch_render(const DeviceScene<R>& ds, const FrameParams<R>& fp, bool cull, R* rgb, int* prim_id, R* dmax,
                          unsigned long long* counters, cudaStream_t stream, const double camera[3] = nullptr,
                          int* launches = nullptr, RenderExtras* extras = nullptr, const ViewBasis* view = nullptr);

// K4: FrameBuffer::normalize + to_vec (framebuffer.rs:40-82) over rows [fp.row_begin, fp.row_end).
template <typename R>
cudaError_t launch_tonemap(const FrameParams<R>& fp, const R* rgb, const R* dmax, bool normalise, unsigned char* rgb8,
                           cudaStream_t stream);

// K4 over the busy tiles of the frame `ds` rendered last with a schedule and RenderExtras::rgb8_zero (same fp).
cudaError_t launch_tonemap_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, const float* dmax,
                                bool normalise, unsigned char* rgb8, cudaStream_t stream);
// The busy tiles of the frame `ds` rendered last with a schedule (same fp): sorted[0] = their number, sorted[1 + k] = the
// k-th in frame order (n_tiles + 1 ints), packed[3072 k ...] = its 32 x 32 x 3 floats.  Two launches.
cudaError_t launch_pack_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, int* sorted, float* packed,
                             cudaStream_t stream);
// ... or written straight into a float32 frame in pinned host memory (device pointer `host_frame`, rows of `host_row_floats`
// floats), tiles [0, n_full) of the schedule's first list and [0, n_busy - n_full) of its second
cudaError_t launch_deliver_busy(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, int n_full, int n_busy,
                                float* host_frame, size_t host_row_floats, cudaStream_t stream);
// launch_tonemap<float> that takes the frame maximum from this rank's mailbox (waiting for every rank's word of frame
// link.seq) and signals rank 0 when its bytes are stored -- the exchange of a rank that has no rows to render (its render
// kernel, which normally does both, is not launched).
cudaError_t launch_tonemap_peer(const DeviceScene<float>& ds, const FrameParams<float>& fp, const float* rgb, const float* dmax,
                                bool normalise, unsigned char* rgb8, cudaStream_t stream, const PeerLink& link);

// resolve_box_kernel: `rows` output rows of `width` pixels (out: rows * width * 3 floats) from the samples x frame `sub`
// (samples * rows rows of samples * width pixels), samples in [1, 8]; *dmax receives max(old, channel maximum of out).
cudaError_t launch_resolve_box(const float* sub, int samples, float* out, int width, int rows, float* dmax, cudaStream_t stream);

// Adaptive anti-aliasing (rm_render_adaptive), three launches after K0 + K1 rendered the 1x frame's rows [lo, hi) into rgb / id:
// adaptive_mark_kernel: rows [row_begin, row_begin + rows) -> mask (1 byte per pixel, from row_begin), the refined pixels
//   appended to list (x | y << 16; *count, zero at launch, receives their number), the unrefined values' maximum into *dmax.
cudaError_t launch_adaptive_mark(const float* rgb, const int* id, int width, int lo, int hi, int row_begin, int rows, float k,
                                 bool all, unsigned char* mask, unsigned* list, unsigned* count, float* dmax, cudaStream_t stream);
// adaptive_subpixel_kernel: the samples^2 sub-pixel values of every listed pixel in the samples x frame fp (sub: 3 samples^2
//   floats per entry), K0's raster records of the same camera reused; *next: a zeroed 64-bit work counter.
cudaError_t launch_adaptive_subpixel(const DeviceScene<float>& ds, const FrameParams<float>& fp, bool cull, int samples,
                                     const unsigned* list, const unsigned* count, unsigned long long* next, float* sub,
                                     const double camera[3], cudaStream_t stream);
// The sampled-frame kernel (rm_sampled.cuh: sampled_kernel<E>), one launcher per effect type E, each in its own translation unit.
// launch_lens (rm_lens.cu, lens_kernel::Effect; rm_render_lens): the n_px output pixels from frame row fp.row_begin of the thin-lens
//   camera lc, each the resolve_box mean of its lc.samples^2 sample rays (rgb: n_px * 3 floats), their maximum into *dmax;
//   *next: a zeroed 64-bit work counter.
cudaError_t launch_lens(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, bool cull, long long n_px,
                        unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream);
// launch_rough_glass (rm_rough.cu, rough_glass_kernel::Effect; rm_render_rough_glass): launch_lens's frame with the reflect / refract
//   recursion turned by the roughness rg (cast_glass_rough); rg.samples == lc.samples.
cudaError_t launch_rough_glass(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const RoughGlass& rg,
                               bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream);
// launch_motion (rm_motion.cu, motion_kernel::Effect; rm_render_motion): launch_lens's frame with every query of sample q at its time
//   mo.tau[q] (MotionView); mo.samples == lc.samples.  ds carries the swept hierarchy; reach = the largest displacement component / 2,
//   by which the primitives leave their uploaded pose (the glass mode's coordinate bound).
cudaError_t launch_motion(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const Motion& mo,
                          double reach, bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax,
                          cudaStream_t stream);
// launch_distributed (rm_distributed.cu, distributed_kernel::Effect; rm_render_distributed): launch_lens's frame with the area lights'
//   one point per sample and level (ap), the rough turn (rg; rg.g null: nothing is rough) and, when `motion`, every query of sample q at its time
//   mo.tau[q] (ds then carries the swept hierarchy, and reach is as for launch_motion); ap, rg and mo have lc.samples.
cudaError_t launch_distributed(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const AreaPoints& ap,
                               const RoughGlass& rg, const Motion& mo, bool motion, double reach, bool cull, long long n_px,
                               unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream);
// launch_indirect (rm_indirect.cu, indirect_kernel::Effect; rm_render_indirect): launch_lens's frame with one diffuse bounce per
//   qualifying opaque hit (cast_indirect) at the disc points df; df.samples == lc.samples.
cudaError_t launch_indirect(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const Diffuse& df,
                            bool cull, long long n_px, unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream);
// launch_path (rm_path.cu, path_kernel::Effect; rm_render_path): launch_distributed's frame with one diffuse bounce per qualifying
//   opaque hit (cast_path) at the disc points df; ap, rg, mo and df have lc.samples, and ds, motion and reach are as for launch_distributed.
cudaError_t launch_path(const DeviceScene<float>& ds, const FrameParams<float>& fp, const LensCamera& lc, const AreaPoints& ap,
                        const RoughGlass& rg, const Motion& mo, const Diffuse& df, bool motion, double reach, bool cull, long long n_px,
                        unsigned long long* next, float* rgb, float* dmax, cudaStream_t stream);
// K0 alone (prepare_raster_kernel, no view): the raster records of `camera` for the kernels that run stage A without K1.
cudaError_t launch_prepare(const DeviceScene<float>& ds, bool cull, const double camera[3], cudaStream_t stream);
// area_light_kernel (rm_area.cu; rm_render_area_lights): after launch_prepare for the same camera, the n_px pixels from frame row
//   fp.row_begin (n_px a multiple of 32): K1's primary hits shaded with the area lights al (rgb: n_px * 3 floats, prim_id:
//   n_px ids or null), their maximum into *dmax; *next: a zeroed 64-bit work counter.
cudaError_t launch_area_lights(const DeviceScene<float>& ds, const FrameParams<float>& fp, const AreaLights& al, bool cull, long long n_px,
                               unsigned long long* next, float* rgb, int* prim_id, float* dmax, const double camera[3], cudaStream_t stream);
// adaptive_resolve_kernel: every listed pixel's resolve_box of its sub-pixel values into rgb (rows from lo), their maximum into
//   *dmax; max_entries bounds *count (sizes the grid).
cudaError_t launch_adaptive_resolve(const float* sub, int samples, const unsigned* list, const unsigned* count, float* rgb, int width,
                                    int lo, long long max_entries, float* dmax, cudaStream_t stream);

// A rank without rows: zero maximum to every mailbox (the others wait for a word of every rank).
cudaError_t launch_publish_zero(const PeerLink& link, float* dmax, cudaStream_t stream);

// Pure-FFMA probe: `iters` x 16 dependent-chain FFMAs per thread on every SM; returns flop count.
cudaError_t launch_ffma_probe(float* sink, int iters, int blocks, cudaStream_t stream, double* flops);

}  // namespace rm
