// rm_api.cu -- implementation of the C ABI declared in include/rm_b200.h.
//
// One process drives one GPU (rm_init(device)).  Scenes are packed on the host (rm_scene.cpp),
// uploaded once and stay resident in HBM; per-frame scratch (float framebuffer, primitive ids,
// RGB8, the max scalar, counters) is cached across calls so the steady-state path allocates
// nothing.  There is no CPU fallback anywhere in this file: every entry point either runs the
// CUDA kernels or returns an error.
#include <cuda_runtime.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rm_b200.h"
#include "rm_kernels.h"
#include "rm_pool.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int fail_cuda(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    cudaGetLastError();         // reported here: a recoverable failure (a refused cudaHostRegister, say) must not surface again
                                // from the next launcher's cudaGetLastError(); a sticky one stays whatever is read
    return (e == cudaErrorMemoryAllocation) ? RM_ERR_OUT_OF_MEMORY : RM_ERR_CUDA;
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call);      \
    } while (0)

// A scene's device memory: ONE allocation (recycled through a small cache: cudaMalloc / cudaFree cost tens of microseconds
// each and cudaFree synchronises the device -- a caller that uploads its scene for every frame, like the reference's
// render() borrowing &Scene, must not pay a dozen of them per frame) filled by ONE host-to-device copy from pinned staging.
struct Arena {
    void* p = nullptr;
    size_t cap = 0;
};
template <typename R> struct DevicePack {
    bool ready = false;
    Arena arena;
    rm::DeviceScene<R> ds;
};

// What the last FP32 render of a scene left behind, for rm_tonemap_device_busy().
struct LastFrame {
    bool classified = false;      // rendered with a tile schedule (K0 classified the tiles: busy ones listed, the rest provably black)
    bool scheduled = false;       // rendered with a tile schedule and the 8-bit frame zero-filled by the render kernel
    int width = 0, height = 0, row_begin = 0, row_step = 0, n_bands = 0, buf_row0 = 0;
    const void* rgb8 = nullptr;
};

struct SceneEntry {
    rm::OwnedFlatScene flat;
    int n_prims = 0;
    DevicePack<float> f32;
    DevicePack<double> f64;
    LastFrame last;
    // A scene's pack holds per-frame mutable state (raster records, frame control block, tile schedule): renders of ONE
    // scene are ordered even when the caller issues them on different streams -- on a change of stream the new stream waits
    // for everything submitted to the previous one.
    bool rendered = false;
    cudaStream_t last_stream = nullptr;
    cudaEvent_t order_ev = nullptr;
    // uploads are asynchronous on the library's stream: the first render after one waits for this event on its own stream
    cudaEvent_t upload_ev = nullptr;
    bool upload_dirty = false;
    // the frame-level call as a CUDA graph (K0 -> K1 with their programmatic launch edge): re-captured per frame -- camera,
    // sequence number and buffers are kernel parameters -- and pushed into the instantiated graph with cudaGraphExecUpdate
    cudaGraphExec_t graph_exec = nullptr;
    long long frames = 0;
};

struct Scratch {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return RM_OK;
        cudaFree(p);
        p = nullptr;
        cap = 0;
        CK(cudaMalloc(&p, bytes));
        cap = bytes;
        return RM_OK;
    }
    void release() { cudaFree(p); p = nullptr; cap = 0; }
};

constexpr int kProfRing = 256;
struct ProfSlot {
    cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};   // before K0, K0|K1, after K1, after K4
    bool has_tone = false;
    bool split = true;                                          // e[1] was recorded between K0 and K1
};

// Pinned host memory owned by the library (staging of the host-delivery path).
struct Pinned {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return RM_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        CK(cudaHostAlloc(&p, bytes, cudaHostAllocDefault));
        cap = bytes;
        return RM_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// What the library last delivered into a caller's frame (rm_render_rows_*, RM_ROWS_RETAINED): which 32x32 tiles hold
// anything but zeros.  Keyed by the address of the frame's first row.
struct Delivered {
    const void* key = nullptr;
    int width = 0, height = 0, elem = 0;
    std::vector<unsigned char> busy;      // per tile of the whole frame: tiles_x * floor(H / 32)
    std::vector<unsigned char> known;     // per 32-row band: the library has delivered it before (its black tiles are black)
};

struct Context {
    bool ready = false;
    int device = -1;
    cudaDeviceProp prop{};
    cudaStream_t stream = nullptr;
    cudaStream_t cap_stream = nullptr;   // frames are captured into their graph here (rm_render_frame)
    long long graph_launches = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // rm_set_profiling: events around K0 / K1 / K4 of every device render, a ring of kProfRing frames
    bool profiling = false;
    std::vector<ProfSlot> prof;
    int prof_head = -1;           // slot of the last recorded frame
    long long prof_frames = 0;    // frames recorded since profiling was switched on
    std::map<RmScene, SceneEntry> scenes;
    RmScene next_handle = 1;
    Scratch rgb, prim, rgb8, small;   // small: [0,8) max scalar, [64, 64+17*8) counters
    Scratch mix;                      // rm_render_dispersive: the frame assembled from the three passes
    Scratch sub;                      // rm_render_supersampled: the s x frame before the resolve; rm_render_adaptive: the
                                      // sub-pixel values of the refined pixels
    Scratch adapt;                    // rm_render_adaptive: the mask bytes and the list of refined pixels
    Scratch pack;                     // host delivery: the busy tiles of a frame, packed in schedule order
    std::vector<Arena> arena_cache;   // device allocations of freed scenes, for the next upload
    // Host packs of the last few scenes by content (SURVEY.md 8f row 2, ingest): a caller that hands over the same scene
    // again -- the reference's render() borrows &Scene for every frame -- gets its pack (sorted primitive classes, raster
    // sources, the hierarchy: 0.1 to 0.2 s for 10^5 primitives) from here and only pays the hash and the upload.
    struct PackEntry {
        uint64_t hash = 0, hash2 = 0;   // two independent 64-bit hashes of the content: a 128-bit key
        size_t bytes = 0;
        std::shared_ptr<rm::PackedScene<float>> pack;
    };
    std::vector<PackEntry> pack_cache;
    Pinned h_upload;                  // pinned staging of a scene upload
    Pinned h_stage, h_order;          // host delivery: pinned staging of the packed tiles / of the tile schedule + counters
    static constexpr int kChunks = 4; // ... the tiles cross PCIe in this many copies, each followed by an event
    cudaEvent_t chunk_ev[kChunks] = {nullptr, nullptr, nullptr, nullptr};
    // ... and the tile schedule is read off the device as soon as K0 has written it, on a stream of its own, so that the
    // host clears the black tiles while K1 renders
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_k0 = nullptr, ev_early = nullptr, ev_list = nullptr;
    Pinned h_early;
    std::unique_ptr<rm::HostPool> pool;
    std::vector<Delivered> delivered; // a handful of frames (RM_ROWS_RETAINED)
    std::mutex mu;
};
Context g;

// A call that writes the caller's float frame [lo, lo + bytes) itself (rm_render_supersampled, rm_render_adaptive): what the
// library last delivered there (RM_ROWS_RETAINED) no longer holds.  A record goes when the frame it describes -- at most
// `height` rows from its key on -- overlaps the bytes written.
void forget_deliveries(const void* lo, size_t bytes) {
    const char* a = static_cast<const char*>(lo);
    const char* b = a + bytes;
    g.delivered.erase(std::remove_if(g.delivered.begin(), g.delivered.end(), [&](const Delivered& d) {
                          const char* k = static_cast<const char*>(d.key);
                          return k < b && k + (size_t)d.height * d.width * 3 * d.elem > a;
                      }), g.delivered.end());
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

int arena_get(size_t bytes, Arena& out) {
    int best = -1;
    for (int i = 0; i < (int)g.arena_cache.size(); i++) {
        const size_t c = g.arena_cache[i].cap;
        if (c >= bytes && c <= 2 * bytes + (1u << 20) && (best < 0 || c < g.arena_cache[best].cap)) best = i;
    }
    if (best >= 0) {
        out = g.arena_cache[best];
        g.arena_cache.erase(g.arena_cache.begin() + best);
        return RM_OK;
    }
    out = Arena();
    const size_t cap = (bytes + 65535) & ~(size_t)65535;
    CK(cudaMalloc(&out.p, cap));
    out.cap = cap;
    return RM_OK;
}
void arena_put(Arena& a) {
    if (!a.p) return;
    if (g.arena_cache.size() >= 8) {
        cudaFree(g.arena_cache.front().p);
        g.arena_cache.erase(g.arena_cache.begin());
    }
    g.arena_cache.push_back(a);
    a = Arena();
}
template <typename R> void release_pack(DevicePack<R>& dp) {
    arena_put(dp.arena);
    dp = DevicePack<R>();
}
// Everything in flight that may read the scene's device memory has finished (before its memory is recycled).
void quiesce_scene(SceneEntry& se) {
    cudaError_t e = cudaSuccess;
    if (se.upload_dirty) e = cudaStreamSynchronize(g.stream);
    if (e == cudaSuccess && se.rendered) e = cudaStreamSynchronize(se.last_stream);
    if (e != cudaSuccess) {                                     // (a caller's stream that no longer exists)
        cudaGetLastError();
        cudaDeviceSynchronize();
    }
}
void destroy_scene(SceneEntry& se) {
    quiesce_scene(se);
    release_pack(se.f32);
    release_pack(se.f64);
    if (se.order_ev) cudaEventDestroy(se.order_ev);
    if (se.upload_ev) cudaEventDestroy(se.upload_ev);
    if (se.graph_exec) cudaGraphExecDestroy(se.graph_exec);
    se.order_ev = se.upload_ev = nullptr;
    se.graph_exec = nullptr;
}

// Called under g.mu before a render of `se` is issued on `stream`.
int order_scene_renders(SceneEntry& se, cudaStream_t stream) {
    if (se.upload_dirty) {
        if (stream != g.stream) CK(cudaStreamWaitEvent(stream, se.upload_ev, 0));
        se.upload_dirty = false;
    }
    if (se.rendered && se.last_stream != stream) {
        if (!se.order_ev) CK(cudaEventCreateWithFlags(&se.order_ev, cudaEventDisableTiming));
        if (cudaEventRecord(se.order_ev, se.last_stream) == cudaSuccess) {
            CK(cudaStreamWaitEvent(stream, se.order_ev, 0));
        } else {                                                // the previous stream is gone: everything it held has been submitted
            cudaGetLastError();
            CK(cudaDeviceSynchronize());
        }
    }
    se.rendered = true;
    se.last_stream = stream;
    return RM_OK;
}

// 64-bit content hash of a byte range: four independent multiply-rotate lanes over 32-byte blocks (memory speed).
uint64_t hash_bytes(const void* data, size_t n, uint64_t seed) {
    const unsigned char* p = static_cast<const unsigned char*>(data);
    uint64_t h[4] = {seed ^ 0x9E3779B97F4A7C15ull, seed ^ 0xC2B2AE3D27D4EB4Full, seed ^ 0x165667B19E3779F9ull, seed ^ 0x27D4EB2F165667C5ull};
    auto mix = [](uint64_t a, uint64_t w) {
        a ^= w * 0x9FB21C651E98DF25ull;
        a = (a << 29) | (a >> 35);
        return a * 0xD6E8FEB86659FD93ull;
    };
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        uint64_t w[4];
        std::memcpy(w, p + i, 32);
        for (int k = 0; k < 4; k++) h[k] = mix(h[k], w[k]);
    }
    uint64_t tail[4] = {0, 0, 0, 0};
    std::memcpy(tail, p + i, n - i);
    for (int k = 0; k < 4; k++) h[k] = mix(h[k], tail[k] ^ (uint64_t)n);
    uint64_t r = h[0] ^ (h[1] << 1 | h[1] >> 63) ^ (h[2] << 2 | h[2] >> 62) ^ (h[3] << 3 | h[3] >> 61);
    r ^= r >> 32;
    return r * 0x9FB21C651E98DF25ull;
}
// Two independent 64-bit content hashes of a flat scene (the key of the pack cache).  Large arrays are hashed in 256 KB
// blocks on the host pool and the block hashes are chained in order: the key does not depend on the number of threads.
rm::HostPool& host_pool();
void hash_scene(const rm::OwnedFlatScene& f, size_t& bytes, uint64_t& h1, uint64_t& h2) {
    constexpr uint64_t kSeed1 = 0x243F6A8885A308D3ull, kSeed2 = 0x13198A2E03707344ull;
    constexpr size_t kBlock = 256 << 10;
    h1 = kSeed1;
    h2 = kSeed2;
    bytes = 0;
    auto add = [&](const auto& v) {
        const size_t n = v.size() * sizeof(v[0]);
        const unsigned char* p = reinterpret_cast<const unsigned char*>(v.data());
        const size_t n_blocks = std::max<size_t>(1, (n + kBlock - 1) / kBlock);
        std::vector<uint64_t> part(2 * n_blocks);
        auto one = [&](int k) {
            const size_t at = (size_t)k * kBlock, len = std::min(kBlock, n - std::min(n, at));
            part[2 * k] = hash_bytes(p + at, len, kSeed1);
            part[2 * k + 1] = hash_bytes(p + at, len, kSeed2);
        };
        if (n_blocks >= 4) host_pool().run((int)n_blocks, one);
        else for (size_t k = 0; k < n_blocks; k++) one((int)k);
        for (size_t k = 0; k < n_blocks; k++) {
            h1 = hash_bytes(&part[2 * k], 8, h1 + v.size());
            h2 = hash_bytes(&part[2 * k + 1], 8, h2 + v.size());
        }
        bytes += n;
    };
    add(f.shapes); add(f.spheres); add(f.polygons); add(f.polygon_vertices); add(f.objs); add(f.triangles);
    add(f.triangle_reflectances); add(f.lights);
}

template <typename R> int pack_for(SceneEntry& se, std::shared_ptr<rm::PackedScene<R>>& out);
template <> int pack_for<double>(SceneEntry& se, std::shared_ptr<rm::PackedScene<double>>& out) {
    out = std::make_shared<rm::PackedScene<double>>();
    std::string err;
    RmFlatScene fs = se.flat.view();
    const int rc = rm::pack_scene<double>(fs, *out, err, &host_pool());
    return rc == RM_OK ? RM_OK : fail(rc, err);
}
template <> int pack_for<float>(SceneEntry& se, std::shared_ptr<rm::PackedScene<float>>& out) {
    size_t bytes = 0;
    uint64_t h = 0, h2 = 0;
    hash_scene(se.flat, bytes, h, h2);
    for (size_t i = 0; i < g.pack_cache.size(); i++)
        if (g.pack_cache[i].hash == h && g.pack_cache[i].hash2 == h2 && g.pack_cache[i].bytes == bytes) {
            out = g.pack_cache[i].pack;
            std::rotate(g.pack_cache.begin() + i, g.pack_cache.begin() + i + 1, g.pack_cache.end());   // most recent last
            return RM_OK;
        }
    out = std::make_shared<rm::PackedScene<float>>();
    std::string err;
    RmFlatScene fs = se.flat.view();
    const int rc = rm::pack_scene<float>(fs, *out, err, &host_pool());
    if (rc != RM_OK) return fail(rc, err);
    if (g.pack_cache.size() >= 4) g.pack_cache.erase(g.pack_cache.begin());
    g.pack_cache.push_back({h, h2, bytes, out});
    return RM_OK;
}

template <typename R> int ensure_pack(SceneEntry& se, DevicePack<R>& dp) {
    if (dp.ready) return RM_OK;
    std::shared_ptr<rm::PackedScene<R>> pack;
    int rc = pack_for<R>(se, pack);
    if (rc != RM_OK) return rc;
    const rm::PackedScene<R>& ps = *pack;
    // layout of the arena: every array at a 256-byte aligned offset, the zero-initialised frame state at the end
    struct Piece { const void* src; size_t bytes, off; };
    std::vector<Piece> pieces;
    size_t total = 0;
    auto add = [&](const void* src, size_t bytes) {
        const size_t off = total;
        pieces.push_back({src, bytes, off});
        total = align256(total + std::max<size_t>(bytes, 16));
        return off;
    };
    auto addv = [&](const auto& v) { return add(v.data(), v.size() * sizeof(v[0])); };
    const size_t o_blob = addv(ps.blob), o_ma = addv(ps.mat_a), o_mb = addv(ps.mat_b), o_mf = addv(ps.mat_f);
    size_t o_ord[2], o_ords[2];
    for (int i = 0; i < 2; i++) {
        o_ord[i] = addv(ps.order[i]);
        o_ords[i] = addv(ps.order_shape[i]);
    }
    size_t o_tsrc = 0, o_nodes = 0, o_prims = 0, o_s64 = 0, o_p64 = 0;
    if (sizeof(R) == 4) {
        o_tsrc = addv(ps.tri_src);
        o_nodes = addv(ps.bvh_nodes);
        o_prims = addv(ps.bvh_prims);
        o_s64 = addv(ps.sph64);
        o_p64 = addv(ps.pln64);
    }
    const size_t copy_bytes = total;
    // FP32 pack: raster records | frame control block | tile schedule | status words of the hierarchy walk, all zero
    const size_t rec_bytes = (size_t)ps.lay.n_tri * 64 + 64;
    const int order_cap = 1 << 16;                              // tiles of a frame up to 8192 x 8192
    const size_t zero_bytes = sizeof(R) == 4 ? rec_bytes + 64 + (size_t)order_cap * sizeof(int) + 64 : 0;
    total = align256(total + zero_bytes);
    if ((rc = arena_get(total, dp.arena)) != RM_OK) return rc;
    // the staging buffer may still feed the previous upload's copy
    CK(cudaStreamSynchronize(g.stream));
    if ((rc = g.h_upload.ensure(copy_bytes)) != RM_OK) return rc;
    char* st = static_cast<char*>(g.h_upload.p);
    for (const Piece& pc : pieces)
        if (pc.bytes) std::memcpy(st + pc.off, pc.src, pc.bytes);
    char* base = static_cast<char*>(dp.arena.p);
    CK(cudaMemcpyAsync(base, st, copy_bytes, cudaMemcpyHostToDevice, g.stream));
    if (zero_bytes) CK(cudaMemsetAsync(base + copy_bytes, 0, zero_bytes, g.stream));
    if (!se.upload_ev) CK(cudaEventCreateWithFlags(&se.upload_ev, cudaEventDisableTiming));
    CK(cudaEventRecord(se.upload_ev, g.stream));
    se.upload_dirty = true;

    for (int i = 0; i < 2; i++) {
        dp.ds.order[i] = reinterpret_cast<const int*>(base + o_ord[i]);
        dp.ds.order_shape[i] = reinterpret_cast<const int*>(base + o_ords[i]);
        dp.ds.n_order[i] = (int)ps.order[i].size();
    }
    if (sizeof(R) == 4) {
        char* z = base + copy_bytes;
        dp.ds.tri_src = reinterpret_cast<const double*>(base + o_tsrc);
        dp.ds.tri_r = reinterpret_cast<rm::R4<float>*>(z);
        dp.ds.ctr = reinterpret_cast<int*>(z + rec_bytes);
        dp.ds.tile_order = dp.ds.ctr + 16;
        dp.ds.tile_order_cap = order_cap;
        dp.ds.bvh.nodes = reinterpret_cast<const rm::R4<float>*>(base + o_nodes);
        dp.ds.bvh.prims = reinterpret_cast<const int*>(base + o_prims);
        dp.ds.bvh.n_nodes = (int)(ps.bvh_nodes.size() / 4);
        dp.ds.bvh.status = dp.ds.tile_order + order_cap;
        dp.ds.sph64 = reinterpret_cast<const double*>(base + o_s64);
        dp.ds.pln64 = reinterpret_cast<const double*>(base + o_p64);
    }
    dp.ds.blob = reinterpret_cast<const unsigned char*>(base + o_blob);
    dp.ds.lay = ps.lay;
    dp.ds.mat_a = reinterpret_cast<const rm::R4<R>*>(base + o_ma);
    dp.ds.mat_b = reinterpret_cast<const rm::R4<R>*>(base + o_mb);
    dp.ds.mat_f = reinterpret_cast<const int*>(base + o_mf);
    dp.ds.n_mat = ps.n_prims;
    se.n_prims = ps.n_prims;
    dp.ready = true;
    return RM_OK;
}

template <typename R> DevicePack<R>& pack_of(SceneEntry& se);
template <> DevicePack<float>& pack_of<float>(SceneEntry& se) { return se.f32; }
template <> DevicePack<double>& pack_of<double>(SceneEntry& se) { return se.f64; }

int check_params(const RmParams* p) {
    if (!p) return fail(RM_ERR_INVALID_ARGUMENT, "params is null");
    if (p->width <= 0 || p->height <= 0) return fail(RM_ERR_INVALID_ARGUMENT, "width and height must be positive");
    if (p->patch_size != 32) return fail(RM_ERR_INVALID_ARGUMENT, "only patch_size 32 is supported (renderer.rs:47)");
    if (p->width % p->patch_size != 0)
        return fail(RM_ERR_DIMENSIONS, "Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)");
    if (p->max_depth < 0 || p->max_depth > rm::kMaxDepth) return fail(RM_ERR_INVALID_ARGUMENT, "max_depth must be in [0, 8]");
    // the production kernel packs pixel coordinates as x | y << 16 in its hit queue and derives tile coordinates with a
    // float reciprocal that is exact below 2^22 tiles
    if (p->width > 65535 || p->height > 65535 || (long long)(p->width / 32) * (p->height / 32) >= (1ll << 22))
        return fail(RM_ERR_DIMENSIONS, "width and height must be below 65536 (and the frame below 2^22 patches)");
    return RM_OK;
}

void fill_counters(RmStats* st, const unsigned long long* c) {
    uint64_t* dst = &st->pixels;
    for (int i = 0; i < rm::C_COUNT; i++) dst[i] = c[i];
}

template <typename R>
int render_device_impl(RmScene scene, const RmParams* params, R* d_rgb, int* d_prim, R* d_max, cudaStream_t stream,
                       int buf_row0_is_tile, unsigned long long* d_counters, rm::FrameParams<R>* out_fp, int* resident,
                       int* launches = nullptr, unsigned char* d_rgb8_zero = nullptr, bool* scheduled = nullptr,
                       const rm::PeerLink* link = nullptr, unsigned char* d_rgb8_out = nullptr, bool normalise = true,
                       unsigned char* d_rgb8_next = nullptr, bool as_graph = false, cudaEvent_t ev_after_k0 = nullptr) {
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    auto it = g.scenes.find(scene);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    DevicePack<R>& dp = pack_of<R>(it->second);
    if ((rc = ensure_pack<R>(it->second, dp)) != RM_OK) return rc;
    if ((rc = order_scene_renders(it->second, stream)) != RM_OK) return rc;
    rm::FrameParams<R> fp = rm::make_frame_params<R>(*params);
    fp.buf_row0 = buf_row0_is_tile ? fp.row_begin : 0;
    if (out_fp) *out_fp = fp;
    const bool cull = params->cull_backfacing != 0;
    if (resident) *resident = dp.ds.lay.n_sph + rm::plane_count<R>(dp.ds.lay, cull);
    rm::RenderExtras ex;
    ex.rgb8_zero = d_rgb8_zero;
    if (link) {
        ex.link = *link;
        ex.zero_dmax = true;
        ex.rgb8_out = d_rgb8_out;
        ex.normalise = normalise;
        ex.rgb8_next = d_rgb8_next;
    }
    if (g.profiling && !g.prof.empty()) {
        g.prof_head = (g.prof_head + 1) % kProfRing;
        g.prof_frames++;
        ProfSlot& ps = g.prof[g.prof_head];
        ps.has_tone = false;
        ps.split = link == nullptr;                             // frame-level calls keep K0 -> K1 a programmatic launch edge
        ex.ev_begin = ps.e[0];
        ex.ev_prepared = ps.split ? ps.e[1] : nullptr;
        ex.ev_rendered = ps.e[2];
    }
    if (ev_after_k0 && !ex.ev_prepared) ex.ev_prepared = ev_after_k0;      // recorded between K0 and K1 (host delivery reads the schedule early)
    SceneEntry& se = it->second;
    // RM_B200_GRAPH=1 (read per call): frame-level calls go to the GPU as ONE graph launch from the scene's second frame on
    // (the first one runs the launchers' one-time set-up).  Opt-in, because on the device it is a wash: 4K cornell frame,
    // alternating blocks of 100 frames, graph against the two launches joined by a programmatic edge: 64.30 / 64.57 us on
    // one box, 64.88 / 64.61 on another, 57.82 / 57.22 at two GPUs (bench.py's graph_ab; profiles/r5m-r5o) -- the edge
    // already hides K1's launch behind K0.  What the graph does save is host time: 40 us instead of 51 us to issue a frame
    // (tools/frame_rate.py), which matters to a caller whose loop is bound by its own thread, not by the GPU.
    // A driver that cannot capture the pair switches it off for the process.
    static int graph_broken = 0;
    const char* genv = getenv("RM_B200_GRAPH");
    const int graph_mode = (!graph_broken && genv && genv[0] == '1') ? 1 : 0;
    bool launched = false;
    if (as_graph && graph_mode == 1 && se.frames > 0 && fp.n_bands > 0) {
        cudaEvent_t ev_begin = ex.ev_begin, ev_rendered = ex.ev_rendered;
        ex.ev_begin = ex.ev_prepared = ex.ev_rendered = nullptr;
        cudaGraph_t graph = nullptr;
        // captured on a stream of the library's own (the caller's may be the legacy default stream, which cannot capture);
        // the graph is launched on the caller's
        cudaError_t e = cudaSuccess;
        if (!g.cap_stream) e = cudaStreamCreateWithFlags(&g.cap_stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamBeginCapture(g.cap_stream, cudaStreamCaptureModeRelaxed);
        if (e == cudaSuccess) {
            const cudaError_t el = rm::launch_render<R>(dp.ds, fp, cull, d_rgb, d_prim, d_max, d_counters, g.cap_stream, params->camera, launches, &ex);
            e = cudaStreamEndCapture(g.cap_stream, &graph);
            if (el != cudaSuccess) e = el;
        }
        if (e == cudaSuccess && se.graph_exec) {
            cudaGraphExecUpdateResultInfo info;
            if (cudaGraphExecUpdate(se.graph_exec, graph, &info) != cudaSuccess) {     // another kernel instantiation (glass mode, layout)
                cudaGetLastError();
                cudaGraphExecDestroy(se.graph_exec);
                se.graph_exec = nullptr;
            }
        }
        if (e == cudaSuccess && !se.graph_exec) e = cudaGraphInstantiate(&se.graph_exec, graph, 0);
        if (e == cudaSuccess) {
            if (ev_begin) cudaEventRecord(ev_begin, stream);
            e = cudaGraphLaunch(se.graph_exec, stream);
            if (ev_rendered) cudaEventRecord(ev_rendered, stream);
        }
        if (graph) cudaGraphDestroy(graph);
        if (e == cudaSuccess) {
            launched = true;
            g.graph_launches++;
        } else {                                                // not on this driver: plain launches from now on
            cudaGetLastError();
            graph_broken = 1;
            if (se.graph_exec) cudaGraphExecDestroy(se.graph_exec);
            se.graph_exec = nullptr;
            ex.ev_begin = ev_begin;
            ex.ev_rendered = ev_rendered;
        }
    }
    if (!launched) CK(rm::launch_render<R>(dp.ds, fp, cull, d_rgb, d_prim, d_max, d_counters, stream, params->camera, launches, &ex));
    se.frames++;
    LastFrame& lf = it->second.last;
    lf.classified = sizeof(R) == 4 && ex.scheduled;
    lf.scheduled = lf.classified && d_rgb8_zero != nullptr;
    lf.width = fp.width; lf.height = fp.height; lf.row_begin = fp.row_begin; lf.row_step = fp.row_step;
    lf.n_bands = fp.n_bands; lf.buf_row0 = fp.buf_row0; lf.rgb8 = d_rgb8_zero;
    if (scheduled) *scheduled = lf.scheduled;
    return RM_OK;
}

template <typename R>
int render_host_impl(RmScene scene, const RmParams* params, R* out_rgb, int32_t* out_prim, uint8_t* out_rgb8, RmStats* stats) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    const bool want_counters = stats && stats->pixels == 1;
    rm::FrameParams<R> fp = rm::make_frame_params<R>(*params);
    // scratch buffers hold the pixel-row span of the call, indexed from its first row (buf_row0 = row_begin)
    const size_t rows = fp.n_bands > 0 ? (size_t)(fp.n_bands - 1) * fp.row_step + 32 : 0;
    const size_t n_px = rows * (size_t)fp.width;
    if ((rc = g.rgb.ensure(std::max<size_t>(n_px * 3 * sizeof(R), 16))) != RM_OK) return rc;
    if (out_prim && (rc = g.prim.ensure(std::max<size_t>(n_px * sizeof(int), 16))) != RM_OK) return rc;
    if (out_rgb8 && (rc = g.rgb8.ensure(std::max<size_t>(n_px * 3, 16))) != RM_OK) return rc;
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    R* d_max = static_cast<R*>(g.small.p);
    unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(static_cast<char*>(g.small.p) + 64);
    cudaStream_t s = g.stream;

    CK(cudaEventRecord(g.ev[0], s));
    CK(cudaMemsetAsync(g.small.p, 0, 1024, s));
    CK(cudaEventRecord(g.ev[1], s));
    int resident = 0;
    int launches = 0;
    bool scheduled = false;
    rc = render_device_impl<R>(scene, params, static_cast<R*>(g.rgb.p), out_prim ? static_cast<int*>(g.prim.p) : nullptr,
                               d_max, s, 1, want_counters ? d_cnt : nullptr, &fp, &resident, &launches,
                               out_rgb8 ? static_cast<unsigned char*>(g.rgb8.p) : nullptr, &scheduled);
    if (rc != RM_OK) return rc;
    CK(cudaEventRecord(g.ev[2], s));
    if (out_rgb8 && rows) {
        if (scheduled) {
            auto it = g.scenes.find(scene);
            CK(rm::launch_tonemap_busy(it->second.f32.ds, reinterpret_cast<const rm::FrameParams<float>&>(fp),
                                       reinterpret_cast<const float*>(g.rgb.p), reinterpret_cast<const float*>(d_max), true,
                                       static_cast<unsigned char*>(g.rgb8.p), s));
        } else {
            CK(rm::launch_tonemap<R>(fp, static_cast<const R*>(g.rgb.p), d_max, true, static_cast<unsigned char*>(g.rgb8.p), s));
        }
        launches++;
    }
    // rendered bands -> host: one copy when they are contiguous, one per 32-row band otherwise
    const int n_copies = fp.row_step == 32 ? (fp.n_bands > 0 ? 1 : 0) : fp.n_bands;
    const size_t band_px = (size_t)(fp.row_step == 32 ? fp.n_bands * 32 : 32) * fp.width;
    for (int b = 0; b < n_copies; b++) {
        const size_t dev_px = (size_t)b * fp.row_step * fp.width;                 // scratch is indexed from row_begin
        const size_t host_px = (size_t)fp.row_begin * fp.width + dev_px;
        if (out_rgb) CK(cudaMemcpyAsync(out_rgb + host_px * 3, static_cast<R*>(g.rgb.p) + dev_px * 3, band_px * 3 * sizeof(R), cudaMemcpyDeviceToHost, s));
        if (out_prim) CK(cudaMemcpyAsync(out_prim + host_px, static_cast<int*>(g.prim.p) + dev_px, band_px * sizeof(int), cudaMemcpyDeviceToHost, s));
        if (out_rgb8) CK(cudaMemcpyAsync(out_rgb8 + host_px * 3, static_cast<unsigned char*>(g.rgb8.p) + dev_px * 3, band_px * 3, cudaMemcpyDeviceToHost, s));
    }
    unsigned char small_host[1024];
    if (stats) CK(cudaMemcpyAsync(small_host, g.small.p, 64 + rm::C_COUNT * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(g.ev[3], s));
    CK(cudaStreamSynchronize(s));
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        if (want_counters) fill_counters(stats, reinterpret_cast<const unsigned long long*>(small_host + 64));
        R mx;
        std::memcpy(&mx, small_host, sizeof(R));
        stats->max_value = (double)mx;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[1], g.ev[2]));
        stats->ms_render = ms;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[3]));
        stats->ms_total = ms;
        stats->kernel_launches = launches;
        stats->resident_prims = resident;
        stats->d2h_bytes = (uint64_t)n_copies * band_px * ((out_rgb ? 3 * sizeof(R) : 0) + (out_prim ? 4 : 0) + (out_rgb8 ? 3 : 0));
    }
    return RM_OK;
}

// ---- host delivery of a frame: what Renderer::render hands back (engine/src/renderer.rs:92-108, framebuffer.rs:6-10) ----
// The caller's frame as row pointers (Vec<Vec<Vec3f>>: one allocation per row) or as one contiguous block.
struct RowSink {
    void* const* rows = nullptr;
    char* base = nullptr;
    size_t row_bytes = 0;
    int elem = 4;                                               // bytes per channel value: 4 (f32) or 8 (f64, the reference's type)
    char* row(int y) const { return rows ? static_cast<char*>(rows[y]) : base + (size_t)y * row_bytes; }
};

// Zero-fill with non-temporal stores: the black part of a frame is written once and not read by these threads, and a
// plain memset of a row segment below the C library's streaming threshold first reads every line it is about to overwrite
// (read-for-ownership) -- twice the memory traffic on a pass that is bound by exactly that.
inline void zero_stream(char* p, size_t n) {
#if defined(__x86_64__)
    while (n && (reinterpret_cast<uintptr_t>(p) & 15)) { *p++ = 0; n--; }
    const __m128i z = _mm_setzero_si128();
    for (; n >= 64; n -= 64, p += 64) {
        _mm_stream_si128(reinterpret_cast<__m128i*>(p), z);
        _mm_stream_si128(reinterpret_cast<__m128i*>(p + 16), z);
        _mm_stream_si128(reinterpret_cast<__m128i*>(p + 32), z);
        _mm_stream_si128(reinterpret_cast<__m128i*>(p + 48), z);
    }
    for (; n >= 16; n -= 16, p += 16) _mm_stream_si128(reinterpret_cast<__m128i*>(p), z);
    while (n) { *p++ = 0; n--; }
#else
    std::memset(p, 0, n);
#endif
}

inline void put_values(char* dst, const float* src, int n, int elem) {
    if (elem == 4) {
        std::memcpy(dst, src, (size_t)n * 4);
    } else {
        double* d = reinterpret_cast<double*>(dst);
        for (int i = 0; i < n; i++) d[i] = (double)src[i];      // exact: the f64 frame holds the FP32 results
    }
}

rm::HostPool& host_pool() {
    if (!g.pool) {
        g.pool.reset(new rm::HostPool(rm::host_thread_count(64)));
    }
    return *g.pool;
}

// FP32 render of the call's bands + delivery into `sink`.  Tile-scheduled frames (triangle-only scenes): the busy tiles
// are packed on the device and cross PCIe in ONE copy (15 MB of the 99 MB cornell frame), the host threads zero-fill the
// provably black tiles while that copy runs and then scatter the busy ones -- with RM_ROWS_RETAINED only the tiles that
// held something in the previous delivery into the same frame and are black now are cleared.  Other scenes: every row
// through the pinned staging buffer (or straight into a contiguous f32 frame).
int render_rows_impl(RmScene scene, const RmParams* params, const RowSink& sink, int flags, RmStats* stats) {
    const auto t_entry = std::chrono::steady_clock::now();
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    if (params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "host delivery of rows computes in RM_FP32 (rm_render_f64 is the RM_FP64 validation call)");
    rm::FrameParams<float> fp = rm::make_frame_params<float>(*params);
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (fp.n_bands <= 0) return RM_OK;
    const int W = fp.width, tiles_x = W / 32, n_tiles = tiles_x * fp.n_bands;
    const size_t span_rows = (size_t)(fp.n_bands - 1) * fp.row_step + 32;
    const size_t n_px = span_rows * (size_t)W;
    if ((rc = g.rgb.ensure(n_px * 12)) != RM_OK) return rc;
    float* d_max = static_cast<float*>(g.small.p);
    cudaStream_t s = g.stream;
    CK(cudaEventRecord(g.ev[0], s));
    CK(cudaMemsetAsync(g.small.p, 0, 64, s));
    CK(cudaEventRecord(g.ev[1], s));
    int resident = 0, launches = 0;
    // (the tile schedule is read off the device right after K0, below: an event between the two launches)
    static const bool early_env = !(getenv("RM_B200_EARLY_SCHEDULE") && getenv("RM_B200_EARLY_SCHEDULE")[0] == '0');
    const bool early_wanted = !g.profiling && early_env;
    if (early_wanted && !g.side_stream) {
        CK(cudaStreamCreateWithFlags(&g.side_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&g.ev_k0, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&g.ev_early, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&g.ev_list, cudaEventDisableTiming));
    }
    rc = render_device_impl<float>(scene, params, static_cast<float*>(g.rgb.p), nullptr, d_max, s, 1, nullptr, &fp, &resident, &launches,
                                   nullptr, nullptr, nullptr, nullptr, true, nullptr, false, early_wanted ? g.ev_k0 : nullptr);
    if (rc != RM_OK) return rc;
    CK(cudaEventRecord(g.ev[2], s));
    SceneEntry& se = g.scenes.find(scene)->second;
    const bool classified = se.last.classified;
    rm::HostPool& pool = host_pool();
    // RM_B200_DELIVERY_TRACE=1: host-side phase times of every delivery on stderr (us since the call's launches were issued)
    static const bool trace = getenv("RM_B200_DELIVERY_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto us_now = [&] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_begin).count(); };
    double t_sched = 0, t_zero = 0, t_copy = 0, t_scatter = 0;
    const int elem = sink.elem;
    const size_t px_bytes = 3 * (size_t)elem;
    float h_max = 0.f;
    uint64_t d2h = 0;

    // the previous delivery into this frame (RM_ROWS_RETAINED)
    const int P = fp.height / 32;
    const void* key = sink.row(fp.row_begin);
    Delivered* prev = nullptr;
    for (auto& d : g.delivered)
        if (d.key == key && d.width == W && d.height == fp.height && d.elem == elem) prev = &d;
    const bool retained = (flags & RM_ROWS_RETAINED) && prev != nullptr;
    if (!prev) {
        if (g.delivered.size() >= 8) g.delivered.erase(g.delivered.begin());
        g.delivered.emplace_back();
        prev = &g.delivered.back();
        prev->key = key; prev->width = W; prev->height = fp.height; prev->elem = elem;
        prev->busy.assign((size_t)tiles_x * P, 0);
        prev->known.assign((size_t)P, 0);
    }

    if (classified) {
        // The schedule as K0 left it -- counters and the two unsorted lists, contiguous in the scene's arena -- crosses on a
        // stream of its own as soon as K0 is done, while K1 renders: the host then knows the busy tiles ~70 us before the
        // sorted list arrives, sizes and issues the tile copies without a synchronisation in the middle of the frame and
        // clears the black tiles while the GPU is still rendering.  The snapshot is only used when it is consistent (K1's last
        // block resets the counters: a snapshot taken after that says so by not adding up) and is checked against the
        // sorted list afterwards.
        const rm::DeviceScene<float>& ds = se.f32.ds;
        const int cap_half = ds.tile_order_cap / 2;
        int early_busy = -1;
        const int* early = nullptr;
        if (early_wanted) {
            const size_t early_ints = 16 + (size_t)cap_half + (size_t)n_tiles;
            if ((rc = g.h_early.ensure(early_ints * sizeof(int))) != RM_OK) return rc;
            CK(cudaStreamWaitEvent(g.side_stream, g.ev_k0, 0));
            CK(cudaMemcpyAsync(g.h_early.p, ds.ctr, early_ints * sizeof(int), cudaMemcpyDeviceToHost, g.side_stream));
            CK(cudaEventRecord(g.ev_early, g.side_stream));
            CK(cudaEventSynchronize(g.ev_early));
            early = static_cast<const int*>(g.h_early.p);
            const int n_full = early[1], n_part = early[5], n_none = early[2];
            if (n_full >= 0 && n_part >= 0 && n_none >= 0 && n_full <= n_tiles && n_part <= n_tiles && n_full + n_part + n_none == n_tiles)
                early_busy = n_full + n_part;
        }
        // A contiguous float32 frame in pinned host memory the device can address is written by the device itself, tile by
        // tile (deliver_busy_kernel): no staging buffer, no scatter.  RM_B200_DIRECT_DELIVERY=0 keeps the staged path.
        float* direct_frame = nullptr;
        static const bool direct_env = !(getenv("RM_B200_DIRECT_DELIVERY") && getenv("RM_B200_DIRECT_DELIVERY")[0] == '0');
        if (direct_env && early_busy >= 0 && elem == 4 && !sink.rows && sink.row_bytes % 16 == 0) {
            char* first = sink.row(fp.row_begin);
            char* last = sink.row(fp.row_begin + (int)span_rows - 1) + (size_t)W * 12 - 1;
            cudaPointerAttributes pa0, pa1;
            if (cudaPointerGetAttributes(&pa0, first) == cudaSuccess && cudaPointerGetAttributes(&pa1, last) == cudaSuccess &&
                pa0.type == cudaMemoryTypeHost && pa1.type == cudaMemoryTypeHost && pa0.devicePointer && pa1.devicePointer &&
                static_cast<char*>(pa1.devicePointer) - static_cast<char*>(pa0.devicePointer) == last - first &&
                (reinterpret_cast<uintptr_t>(pa0.devicePointer) & 15) == 0)
                direct_frame = reinterpret_cast<float*>(static_cast<char*>(pa0.devicePointer) - (size_t)fp.row_begin * sink.row_bytes);
            else
                cudaGetLastError();                             // (pageable memory: not an error, the staged path takes it)
        }
        // device: [sorted list: n_tiles + 1 ints][packed tiles]; host (pinned): the same list, then the tiles
        const size_t list_bytes = align256((size_t)(n_tiles + 1) * sizeof(int));
        if ((rc = g.h_order.ensure(list_bytes + 64)) != RM_OK) return rc;
        int* h_sorted = static_cast<int*>(g.h_order.p);
        float* h_maxp = reinterpret_cast<float*>(static_cast<char*>(g.h_order.p) + list_bytes);
        int* d_sorted = nullptr;
        float* d_packed = nullptr;
        if (direct_frame) {
            CK(rm::launch_deliver_busy(ds, fp, static_cast<const float*>(g.rgb.p), early[1], early_busy, direct_frame, sink.row_bytes / 4, s));
            launches += 1;
            CK(cudaMemcpyAsync(h_maxp, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
        } else {
            if ((rc = g.pack.ensure(list_bytes + (size_t)n_tiles * 12288)) != RM_OK) return rc;
            d_sorted = static_cast<int*>(g.pack.p);
            d_packed = reinterpret_cast<float*>(static_cast<char*>(g.pack.p) + list_bytes);
            CK(rm::launch_pack_busy(ds, fp, static_cast<const float*>(g.rgb.p), d_sorted, d_packed, s));
            launches += 2;
            CK(cudaMemcpyAsync(h_sorted, d_sorted, (size_t)(n_tiles + 1) * sizeof(int), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(h_maxp, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
            if (early_wanted) CK(cudaEventRecord(g.ev_list, s));
        }
        int n_busy = early_busy;
        const int* tiles = h_sorted + 1;
        if (n_busy < 0) {                                        // no snapshot: wait for the sorted list
            CK(cudaStreamSynchronize(s));
            n_busy = h_sorted[0];
            h_max = *h_maxp;
            if (n_busy < 0 || n_busy > n_tiles) return fail(RM_ERR_CUDA, "tile schedule of the frame is inconsistent");
        }
        t_sched = us_now();
        if (!direct_frame && (rc = g.h_stage.ensure(std::max<size_t>((size_t)n_busy * 12288, 64))) != RM_OK) return rc;
        // the busy tiles cross PCIe in a few chunks, each followed by an event: the host scatters chunk k while chunk
        // k + 1 is still on its way (one cudaMemcpyAsync per chunk)
        constexpr int kChunks = Context::kChunks;
        cudaEvent_t* const chunk_ev = g.chunk_ev;
        int chunk_end[kChunks];
        int n_chunks = 0;
        for (int k = 0; k < kChunks && n_busy > 0 && !direct_frame; k++) {
            const int a0 = (int)((long long)n_busy * k / kChunks), a1 = (int)((long long)n_busy * (k + 1) / kChunks);
            if (a1 <= a0) continue;
            if (!chunk_ev[n_chunks]) CK(cudaEventCreateWithFlags(&chunk_ev[n_chunks], cudaEventDisableTiming));
            CK(cudaMemcpyAsync(static_cast<char*>(g.h_stage.p) + (size_t)a0 * 12288, reinterpret_cast<const char*>(d_packed) + (size_t)a0 * 12288,
                               (size_t)(a1 - a0) * 12288, cudaMemcpyDeviceToHost, s));
            CK(cudaEventRecord(chunk_ev[n_chunks], s));
            chunk_end[n_chunks++] = a1;
        }
        CK(cudaEventRecord(g.ev[3], s));
        d2h = (uint64_t)n_busy * 12288 + (direct_frame ? 0 : (uint64_t)(n_tiles + 1) * sizeof(int)) + 4;
        // while they travel: which tiles are busy now, and the black ones cleared
        std::vector<unsigned char> now((size_t)n_tiles, 0);
        if (early_busy >= 0) {
            d2h += (uint64_t)(16 + cap_half + n_tiles) * sizeof(int);
            const int n_full = early[1];
            for (int t = 0; t < n_busy; t++) {
                const int tile = t < n_full ? early[16 + t] : early[16 + cap_half + (t - n_full)];
                if (tile < 0 || tile >= n_tiles || now[tile]) return fail(RM_ERR_CUDA, "tile schedule of the frame is inconsistent");
                now[tile] = 1;
            }
        } else {
            for (int t = 0; t < n_busy; t++) {
                if (tiles[t] < 0 || tiles[t] >= n_tiles || (t && tiles[t] <= tiles[t - 1])) return fail(RM_ERR_CUDA, "tile schedule of the frame is inconsistent");
                now[tiles[t]] = 1;
            }
        }
        const int band0 = fp.row_begin / 32, band_step = fp.row_step / 32;
        unsigned char* pb = prev->busy.data();
        // per pixel row of the call's bands: a band the library has not delivered into this frame before (or any band
        // without RM_ROWS_RETAINED) gets every black tile cleared, runs of black tiles in one memset; a known band only
        // the tiles that held something in the previous delivery and are black now
        bool any_clear = !retained;
        for (int b = 0; b < fp.n_bands && !any_clear; b++) {
            const int band = band0 + b * band_step;
            if (!prev->known[band]) any_clear = true;
            for (int tx = 0; tx < tiles_x && !any_clear; tx++) any_clear = pb[(size_t)band * tiles_x + tx] && !now[(size_t)b * tiles_x + tx];
        }
        if (any_clear)
            pool.run(fp.n_bands * 32, [&](int item) {
                const int b = item >> 5, r = item & 31, band = band0 + b * band_step;
                char* row = sink.row(fp.row_begin + b * fp.row_step + r);
                const unsigned char* nb = now.data() + (size_t)b * tiles_x;
                const unsigned char* ob = pb + (size_t)band * tiles_x;
                const bool delta = retained && prev->known[band];
                for (int tx = 0; tx < tiles_x;) {
                    if (nb[tx] || (delta && !ob[tx])) { tx++; continue; }
                    int e = tx + 1;
                    while (e < tiles_x && !nb[e] && !(delta && !ob[e])) e++;
                    zero_stream(row + (size_t)tx * 32 * px_bytes, (size_t)(e - tx) * 32 * px_bytes);
                    tx = e;
                }
#if defined(__x86_64__)
                _mm_sfence();
#endif
            });
        for (int b = 0; b < fp.n_bands; b++) {
            prev->known[band0 + b * band_step] = 1;
            std::memcpy(pb + (size_t)(band0 + b * band_step) * tiles_x, now.data() + (size_t)b * tiles_x, tiles_x);
        }
        if (direct_frame) {
            CK(cudaStreamSynchronize(s));                       // the device has written the busy tiles into the caller's frame
            h_max = *h_maxp;
            t_copy = us_now();
        } else if (early_busy >= 0) {
            // the sorted list (the order the tiles were packed in) and the maximum have arrived long since: same tiles?
            CK(cudaEventSynchronize(g.ev_list));
            h_max = *h_maxp;
            bool same = h_sorted[0] == n_busy;
            for (int t = 0; t < n_busy && same; t++) same = tiles[t] >= 0 && tiles[t] < n_tiles && now[tiles[t]] && (!t || tiles[t] > tiles[t - 1]);
            if (!same) return fail(RM_ERR_CUDA, "tile schedule of the frame is inconsistent");
        }
        t_zero = us_now();
        // scatter, chunk by chunk; an item is a run of up to 8 tiles in frame order -- neighbours in a band share the pages
        // of their 32 pixel rows, so a thread walks row by row over the run
        const float* stage = static_cast<const float*>(g.h_stage.p);
        int done = 0;
        for (int k = 0; k < n_chunks; k++) {
            CK(cudaEventSynchronize(chunk_ev[k]));
            if (k == n_chunks - 1) t_copy = us_now();
            const int c0 = done, c1 = chunk_end[k];
            pool.run((c1 - c0 + 7) / 8, [&](int item) {
                const int t0 = c0 + item * 8, t1 = std::min(t0 + 8, c1);
                for (int r = 0; r < 32; r++)
                    for (int t = t0; t < t1; t++) {
                        const int tile = tiles[t], ty = tile / tiles_x, tx = tile - ty * tiles_x;
                        put_values(sink.row(fp.row_begin + ty * fp.row_step + r) + (size_t)tx * 32 * px_bytes,
                                   stage + (size_t)t * 3072 + r * 96, 96, elem);
                    }
            }, 8);
            done = c1;
        }
        t_scatter = us_now();
        if (trace)
            std::fprintf(stderr, "rm delivery: %d busy of %d tiles, %s: launches issued %.0f us after entry; from there: schedule on host %.0f us, black tiles cleared %.0f, copy done %.0f, scattered %.0f (%d threads)\n",
                         n_busy, n_tiles, retained ? "retained" : "fresh", std::chrono::duration<double, std::micro>(t_begin - t_entry).count(),
                         t_sched, t_zero, t_copy, t_scatter, pool.threads());
    } else {
        // no schedule (spheres, n-gons, hierarchy): every rendered row holds something
        const bool direct = elem == 4 && !sink.rows && sink.row_bytes == (size_t)W * 12;
        const size_t band_bytes = (size_t)32 * W * 12;
        if (!direct && (rc = g.h_stage.ensure((size_t)fp.n_bands * band_bytes)) != RM_OK) return rc;
        for (int b = 0; b < fp.n_bands; b++) {
            const char* src = static_cast<const char*>(g.rgb.p) + (size_t)b * fp.row_step * W * 12;
            char* dst = direct ? sink.row(fp.row_begin + b * fp.row_step) : static_cast<char*>(g.h_stage.p) + (size_t)b * band_bytes;
            const size_t n = (direct && fp.row_step == 32) ? band_bytes * fp.n_bands : band_bytes;
            CK(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, s));
            d2h += n;
            if (direct && fp.row_step == 32) break;
        }
        CK(cudaMemcpyAsync(&h_max, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
        CK(cudaEventRecord(g.ev[3], s));
        CK(cudaStreamSynchronize(s));
        if (!direct) {
            const float* stage = static_cast<const float*>(g.h_stage.p);
            pool.run(fp.n_bands * 32, [&](int item) {
                const int b = item >> 5, r = item & 31;
                put_values(sink.row(fp.row_begin + b * fp.row_step + r), stage + ((size_t)b * 32 + r) * W * 3, W * 3, elem);
            });
        }
        const int band0 = fp.row_begin / 32, band_step = fp.row_step / 32;
        for (int b = 0; b < fp.n_bands; b++) {
            std::memset(prev->busy.data() + (size_t)(band0 + b * band_step) * tiles_x, 1, tiles_x);
            prev->known[band0 + b * band_step] = 1;
        }
    }
    if (stats) {
        stats->max_value = (double)h_max;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[1], g.ev[2]));
        stats->ms_render = ms;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[3]));
        stats->ms_total = ms;
        stats->kernel_launches = launches;
        stats->resident_prims = resident;
        stats->d2h_bytes = d2h;
    }
    return RM_OK;
}

}  // namespace

extern "C" {

int rm_abi_version(void) { return RM_ABI_VERSION; }

const char* rm_last_error(void) { return g_err.c_str(); }

int rm_init(int device) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (g.ready && g.device == device) return RM_OK;
    if (g.ready) return fail(RM_ERR_INVALID_ARGUMENT, "already initialised on another device; call rm_shutdown() first");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_err = std::string("no CUDA device available: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                " -- this library has no CPU fallback";
        return RM_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) return fail(RM_ERR_NO_DEVICE, "device ordinal out of range");
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail_cuda(e, "cudaSetDevice"), RM_ERR_NO_DEVICE;
    if ((e = cudaGetDeviceProperties(&g.prop, device)) != cudaSuccess) return fail_cuda(e, "cudaGetDeviceProperties"), RM_ERR_NO_DEVICE;
    if (g.prop.major != 10) {
        char buf[256];
        std::snprintf(buf, sizeof buf, "device %d (%s) is sm_%d%d; the kernels are built for sm_100a only", device, g.prop.name,
                      g.prop.major, g.prop.minor);
        return fail(RM_ERR_NO_DEVICE, buf);
    }
    CK(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    for (auto& ev : g.ev) CK(cudaEventCreate(&ev));
    g.device = device;
    g.ready = true;
    return RM_OK;
}

void rm_shutdown(void) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return;
    cudaSetDevice(g.device);
    cudaDeviceSynchronize();
    for (auto& kv : g.scenes) destroy_scene(kv.second);
    g.scenes.clear();
    for (auto& a : g.arena_cache) cudaFree(a.p);
    g.arena_cache.clear();
    g.pack_cache.clear();
    g.rgb.release(); g.prim.release(); g.rgb8.release(); g.small.release(); g.mix.release(); g.pack.release(); g.sub.release(); g.adapt.release();
    g.h_stage.release(); g.h_order.release(); g.h_upload.release(); g.h_early.release();
    if (g.side_stream) cudaStreamDestroy(g.side_stream);
    g.side_stream = nullptr;
    for (cudaEvent_t* ev : {&g.ev_k0, &g.ev_early, &g.ev_list}) { if (*ev) cudaEventDestroy(*ev); *ev = nullptr; }
    g.pool.reset();
    g.delivered.clear();
    for (auto& ev : g.chunk_ev) { if (ev) cudaEventDestroy(ev); ev = nullptr; }
    for (auto& ev : g.ev) { if (ev) cudaEventDestroy(ev); ev = nullptr; }
    for (auto& ps : g.prof)
        for (auto& ev : ps.e) { if (ev) cudaEventDestroy(ev); ev = nullptr; }
    g.prof.clear();
    g.profiling = false;
    g.prof_head = -1;
    g.prof_frames = 0;
    if (g.stream) cudaStreamDestroy(g.stream);
    g.stream = nullptr;
    if (g.cap_stream) cudaStreamDestroy(g.cap_stream);
    g.cap_stream = nullptr;
    g.graph_launches = 0;
    g.ready = false;
    g.device = -1;
}

int rm_device_info(char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz) {
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (name && name_len > 0) { std::strncpy(name, g.prop.name, name_len - 1); name[name_len - 1] = 0; }
    if (sm_count) *sm_count = g.prop.multiProcessorCount;
    if (cc_major) *cc_major = g.prop.major;
    if (cc_minor) *cc_minor = g.prop.minor;
    if (clock_khz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g.device);
        *clock_khz = khz;
    }
    return RM_OK;
}

void rm_params_default(RmParams* p, int width, int height) {
    std::memset(p, 0, sizeof(*p));
    p->width = width;
    p->height = height;
    p->fov = 1.5;            // main.rs:368
    p->max_depth = 3;        // renderer.rs:262
    p->background = 0.1;     // renderer.rs:40-44
    p->patch_size = 32;      // renderer.rs:47
    p->precision = RM_FP32;
    p->patch_row_begin = 0;
    p->patch_row_end = -1;
    p->cull_backfacing = 1;
    p->patch_row_stride = 1;
}

int rm_scene_upload(const RmFlatScene* scene, RmScene* out_handle) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    if (!scene || !out_handle) return fail(RM_ERR_INVALID_ARGUMENT, "scene or out_handle is null");
    std::string err;
    int rc = rm::validate_scene(*scene, err);
    if (rc != RM_OK) return fail(rc, err);
    SceneEntry se;
    se.flat.assign(*scene, &host_pool());
    if ((rc = ensure_pack<float>(se, se.f32)) != RM_OK) { destroy_scene(se); return rc; }
    RmScene h = g.next_handle++;
    g.scenes.emplace(h, std::move(se));
    *out_handle = h;
    return RM_OK;
}

int rm_scene_free(RmScene handle) {
    std::lock_guard<std::mutex> lock(g.mu);
    auto it = g.scenes.find(handle);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    destroy_scene(it->second);                                  // waits for the scene's renders, recycles its device memory
    g.scenes.erase(it);
    return RM_OK;
}

int rm_scene_num_prims(RmScene handle) {
    std::lock_guard<std::mutex> lock(g.mu);
    auto it = g.scenes.find(handle);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    return it->second.n_prims;
}

int rm_render(RmScene scene, const RmParams* params, float* out_rgb, int32_t* out_prim_id, uint8_t* out_rgb8, RmStats* stats) {
    if (params && params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render computes in RM_FP32; use rm_render_f64 for RM_FP64");
    if (out_rgb && !out_prim_id && !out_rgb8 && params && !(stats && stats->pixels == 1)) {
        // the float frame only -- what Renderer::render returns: the packed host delivery (bit-identical rows)
        RowSink sink;
        sink.base = reinterpret_cast<char*>(out_rgb);
        sink.row_bytes = (size_t)std::max(params->width, 0) * 12;
        sink.elem = 4;
        return render_rows_impl(scene, params, sink, 0, stats);
    }
    return render_host_impl<float>(scene, params, out_rgb, out_prim_id, out_rgb8, stats);
}

namespace {
// Row pointers that turn out to be one contiguous block (a frame kept as one allocation) are treated as such: rows can
// then be copied from the device straight into the caller's memory when nothing has to be widened or scattered.
RowSink sink_of_rows(void* const* rows, const RmParams* params, int elem) {
    RowSink sink;
    sink.rows = rows;
    sink.elem = elem;
    if (params && params->width > 0 && params->height > 0) {
        const size_t row_bytes = (size_t)params->width * 3 * elem;
        bool contiguous = true;
        for (int y = 1; y < params->height && contiguous; y++)
            contiguous = static_cast<const char*>(rows[y]) == static_cast<const char*>(rows[y - 1]) + row_bytes;
        if (contiguous) {
            sink.rows = nullptr;
            sink.base = static_cast<char*>(rows[0]);
            sink.row_bytes = row_bytes;
        }
    }
    return sink;
}
}  // namespace

int rm_render_rows_f32(RmScene scene, const RmParams* params, float* const* rows, int flags, RmStats* stats) {
    if (!rows) return fail(RM_ERR_INVALID_ARGUMENT, "rows is null");
    return render_rows_impl(scene, params, sink_of_rows(reinterpret_cast<void* const*>(rows), params, 4), flags, stats);
}

int rm_render_rows_f64(RmScene scene, const RmParams* params, double* const* rows, int flags, RmStats* stats) {
    if (!rows) return fail(RM_ERR_INVALID_ARGUMENT, "rows is null");
    return render_rows_impl(scene, params, sink_of_rows(reinterpret_cast<void* const*>(rows), params, 8), flags, stats);
}

int rm_render_f64(RmScene scene, const RmParams* params, double* out_rgb, int32_t* out_prim_id, uint8_t* out_rgb8, RmStats* stats) {
    return render_host_impl<double>(scene, params, out_rgb, out_prim_id, out_rgb8, stats);
}

// Extension mode (include/rm_b200.h): three passes of the unchanged render kernels, channel c of pass c kept.  The merge
// is three pitched device-to-device copies (one float of every pixel: width 4 bytes, pitch 12) -- no kernel of its own.
int rm_render_dispersive(const RmScene scenes[3], const RmParams* params, float* out_rgb, int32_t* out_prim_id, RmStats* stats) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    if (!scenes) return fail(RM_ERR_INVALID_ARGUMENT, "scenes is null");
    if (params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_dispersive computes in RM_FP32");
    if (params->patch_row_stride > 1) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_dispersive renders contiguous patch rows (patch_row_stride <= 1)");
    rm::FrameParams<float> fp = rm::make_frame_params<float>(*params);
    const size_t rows = (size_t)fp.n_bands * 32;
    const size_t n_px = rows * (size_t)fp.width;
    if ((rc = g.rgb.ensure(std::max<size_t>(n_px * 12, 16))) != RM_OK) return rc;
    if ((rc = g.mix.ensure(std::max<size_t>(n_px * 12, 16))) != RM_OK) return rc;
    if (out_prim_id && (rc = g.prim.ensure(std::max<size_t>(n_px * sizeof(int), 16))) != RM_OK) return rc;
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    float* d_max = static_cast<float*>(g.small.p);
    cudaStream_t s = g.stream;
    CK(cudaEventRecord(g.ev[0], s));
    int resident = 0, launches = 0;
    for (int c = 0; c < 3; c++) {
        CK(cudaMemsetAsync(g.small.p, 0, 1024, s));
        // (the primary ray does not depend on the refractive index: the ids of the first pass are the frame's)
        rc = render_device_impl<float>(scenes[c], params, static_cast<float*>(g.rgb.p), (out_prim_id && c == 0) ? static_cast<int*>(g.prim.p) : nullptr,
                                       d_max, s, 1, nullptr, nullptr, &resident, &launches);
        if (rc != RM_OK) return rc;
        if (n_px)
            CK(cudaMemcpy2DAsync(static_cast<char*>(g.mix.p) + 4 * c, 12, static_cast<const char*>(g.rgb.p) + 4 * c, 12, 4, n_px,
                                 cudaMemcpyDeviceToDevice, s));
    }
    CK(cudaEventRecord(g.ev[2], s));
    const size_t host_px = (size_t)fp.row_begin * fp.width;
    if (out_rgb && n_px) CK(cudaMemcpyAsync(out_rgb + host_px * 3, g.mix.p, n_px * 12, cudaMemcpyDeviceToHost, s));
    if (out_prim_id && n_px) CK(cudaMemcpyAsync(out_prim_id + host_px, g.prim.p, n_px * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(g.ev[3], s));
    CK(cudaStreamSynchronize(s));
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[2]));
        stats->ms_render = ms;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[3]));
        stats->ms_total = ms;
        stats->kernel_launches = launches;
        stats->resident_prims = resident;
    }
    return RM_OK;
}

// Extension mode (include/rm_b200.h): the unchanged render kernels on the s x frame into a scratch of its own, then
// resolve_box_kernel (the W-wide rows and their maximum) and, for the 8-bit frame, the tone-map kernel.
int rm_render_supersampled(RmScene scene, const RmParams* params, int samples, float* out_rgb, uint8_t* out_rgb8, RmStats* stats) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    if (samples < 1 || samples > 8) return fail(RM_ERR_INVALID_ARGUMENT, "samples must be in [1, 8]");
    if (params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_supersampled computes in RM_FP32");
    if (params->patch_row_stride > 1) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_supersampled renders contiguous patch rows (patch_row_stride <= 1)");
    if (g.scenes.find(scene) == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    if (!out_rgb && !out_rgb8) return fail(RM_ERR_INVALID_ARGUMENT, "out_rgb and out_rgb8 are both null");
    rm::FrameParams<float> fp = rm::make_frame_params<float>(*params);
    fp.buf_row0 = fp.row_begin;                                 // the scratch frames are indexed from the call's first row
    // the s x frame renders exactly the sub-rows of the call's patch rows [b, e): its patch rows [s b, s e)
    RmParams sp = *params;
    sp.width = samples * params->width;
    sp.height = samples * params->height;
    sp.patch_row_begin = samples * (fp.row_begin / 32);
    sp.patch_row_end = samples * (fp.row_end / 32);
    sp.patch_row_stride = 1;
    if ((rc = check_params(&sp)) != RM_OK) return rc;
    const size_t rows = (size_t)fp.n_bands * 32, n_px = rows * (size_t)fp.width;
    if ((rc = g.sub.ensure(std::max<size_t>(n_px * samples * samples * 12, 16))) != RM_OK) return rc;
    if ((rc = g.rgb.ensure(std::max<size_t>(n_px * 12, 16))) != RM_OK) return rc;
    if (out_rgb8 && (rc = g.rgb8.ensure(std::max<size_t>(n_px * 3, 16))) != RM_OK) return rc;
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    float* d_max = static_cast<float*>(g.small.p);              // of the resolved rows
    float* d_sub_max = d_max + 2;                               // of the s x frame (not reported)
    cudaStream_t s = g.stream;
    CK(cudaEventRecord(g.ev[0], s));
    CK(cudaMemsetAsync(g.small.p, 0, 64, s));
    CK(cudaEventRecord(g.ev[1], s));
    int resident = 0, launches = 0;
    rc = render_device_impl<float>(scene, &sp, static_cast<float*>(g.sub.p), nullptr, d_sub_max, s, 1, nullptr, nullptr, &resident, &launches);
    if (rc != RM_OK) return rc;
    CK(cudaEventRecord(g.ev[2], s));
    if (rows) {
        CK(rm::launch_resolve_box(static_cast<const float*>(g.sub.p), samples, static_cast<float*>(g.rgb.p), fp.width, (int)rows, d_max, s));
        launches++;
        if (out_rgb8) {
            CK(rm::launch_tonemap<float>(fp, static_cast<const float*>(g.rgb.p), d_max, true, static_cast<unsigned char*>(g.rgb8.p), s));
            launches++;
        }
    }
    const size_t host_px = (size_t)fp.row_begin * fp.width;
    if (out_rgb && n_px) {
        forget_deliveries(out_rgb + host_px * 3, n_px * 12);
        CK(cudaMemcpyAsync(out_rgb + host_px * 3, g.rgb.p, n_px * 12, cudaMemcpyDeviceToHost, s));
    }
    if (out_rgb8 && n_px) CK(cudaMemcpyAsync(out_rgb8 + host_px * 3, g.rgb8.p, n_px * 3, cudaMemcpyDeviceToHost, s));
    float h_max = 0.f;
    if (stats) CK(cudaMemcpyAsync(&h_max, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(g.ev[3], s));
    CK(cudaStreamSynchronize(s));
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->max_value = (double)h_max;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[1], g.ev[2]));
        stats->ms_render = ms;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[3]));
        stats->ms_total = ms;
        stats->kernel_launches = launches;
        stats->resident_prims = resident;
        stats->d2h_bytes = (uint64_t)n_px * ((out_rgb ? 12 : 0) + (out_rgb8 ? 3 : 0));
    }
    return RM_OK;
}

// Extension mode (include/rm_b200.h): the unchanged render kernels on the 1x frame of the call's rows plus one patch row
// of halo on either side, adaptive_mark_kernel (mask, list of refined pixels, maximum of the others), adaptive_subpixel_kernel
// (the s x frame's sub-pixels of the listed pixels only), adaptive_resolve_kernel over the list and, for the 8-bit frame,
// the tone-map kernel.  The list length stays on the device: no host round trip between the launches.
int rm_render_adaptive(RmScene scene, const RmParams* params, int samples, double contrast, float* out_rgb, uint8_t* out_rgb8,
                       uint8_t* out_mask, RmStats* stats) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    if (samples < 1 || samples > 8) return fail(RM_ERR_INVALID_ARGUMENT, "samples must be in [1, 8]");
    if (contrast != contrast) return fail(RM_ERR_INVALID_ARGUMENT, "contrast is NaN");
    if (params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_adaptive computes in RM_FP32");
    if (params->patch_row_stride > 1) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_adaptive renders contiguous patch rows (patch_row_stride <= 1)");
    if (params->max_depth < 1) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_adaptive needs max_depth >= 1");
    auto it = g.scenes.find(scene);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    if (!out_rgb && !out_rgb8) return fail(RM_ERR_INVALID_ARGUMENT, "out_rgb and out_rgb8 are both null");
    const rm::FrameParams<float> fp = rm::make_frame_params<float>(*params);      // the output rows [row_begin, row_end)
    // the s x frame, whose sub-pixels the refined pixels get: only its FrameParams are used, but it must be a valid frame
    RmParams sp = *params;
    sp.width = samples * params->width;
    sp.height = samples * params->height;
    sp.patch_row_begin = 0;
    sp.patch_row_end = -1;
    sp.patch_row_stride = 1;
    if ((rc = check_params(&sp)) != RM_OK) return rc;
    const rm::FrameParams<float> fs = rm::make_frame_params<float>(sp);
    // the 1x frame: the call's patch rows and one more above and below where the frame has one (the mask's neighbours)
    const int b = fp.row_begin / 32, e = fp.row_end / 32;
    RmParams hp = *params;
    hp.patch_row_begin = e > b ? std::max(b - 1, 0) : b;
    hp.patch_row_end = e > b ? std::min(e + 1, params->height / 32) : b;
    hp.patch_row_stride = 1;
    const int lo = 32 * hp.patch_row_begin, hi = 32 * hp.patch_row_end;
    const size_t halo_px = (size_t)(hi - lo) * fp.width, rows = (size_t)fp.n_bands * 32, n_px = rows * (size_t)fp.width;
    const size_t ss = (size_t)samples * samples;
    if ((rc = g.rgb.ensure(std::max<size_t>(halo_px * 12, 16))) != RM_OK) return rc;
    if ((rc = g.prim.ensure(std::max<size_t>(halo_px * 4, 16))) != RM_OK) return rc;
    if (out_rgb8 && (rc = g.rgb8.ensure(std::max<size_t>(halo_px * 3, 16))) != RM_OK) return rc;
    if ((rc = g.sub.ensure(std::max<size_t>(n_px * ss * 12, 16))) != RM_OK) return rc;
    const size_t list_off = align256(n_px);
    if ((rc = g.adapt.ensure(std::max<size_t>(list_off + n_px * 4, 16))) != RM_OK) return rc;
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    float* d_max = static_cast<float*>(g.small.p);              // of the output rows
    float* d_max1 = d_max + 2;                                  // of the 1x frame with its halo (not reported)
    unsigned* d_count = reinterpret_cast<unsigned*>(static_cast<char*>(g.small.p) + 16);
    unsigned long long* d_next = reinterpret_cast<unsigned long long*>(static_cast<char*>(g.small.p) + 24);
    unsigned char* d_mask = static_cast<unsigned char*>(g.adapt.p);
    unsigned* d_list = reinterpret_cast<unsigned*>(static_cast<char*>(g.adapt.p) + list_off);
    float* d_rgb = static_cast<float*>(g.rgb.p);
    const size_t dev_px = (size_t)(fp.row_begin - lo) * fp.width;     // first output pixel in the 1x scratch
    cudaStream_t s = g.stream;
    CK(cudaEventRecord(g.ev[0], s));
    CK(cudaMemsetAsync(g.small.p, 0, 64, s));
    CK(cudaEventRecord(g.ev[1], s));
    int resident = 0, launches = 0;
    rc = render_device_impl<float>(scene, &hp, d_rgb, static_cast<int*>(g.prim.p), d_max1, s, 1, nullptr, nullptr, &resident, &launches);
    if (rc != RM_OK) return rc;
    if (rows) {
        CK(rm::launch_adaptive_mark(d_rgb, static_cast<const int*>(g.prim.p), fp.width, lo, hi, fp.row_begin, (int)rows, (float)contrast,
                                    contrast < 0., d_mask, d_list, d_count, d_max, s));
        CK(rm::launch_adaptive_subpixel(it->second.f32.ds, fs, params->cull_backfacing != 0, samples, d_list, d_count, d_next,
                                        static_cast<float*>(g.sub.p), params->camera, s));
        CK(rm::launch_adaptive_resolve(static_cast<const float*>(g.sub.p), samples, d_list, d_count, d_rgb, fp.width, lo, (long long)n_px,
                                       d_max, s));
        launches += 3;
    }
    CK(cudaEventRecord(g.ev[2], s));
    if (out_rgb8 && rows) {
        rm::FrameParams<float> fo = fp;
        fo.buf_row0 = lo;                                       // both scratch frames are indexed from the halo's first row
        CK(rm::launch_tonemap<float>(fo, d_rgb, d_max, true, static_cast<unsigned char*>(g.rgb8.p), s));
        launches++;
    }
    const size_t host_px = (size_t)fp.row_begin * fp.width;
    if (out_rgb && n_px) {
        forget_deliveries(out_rgb + host_px * 3, n_px * 12);
        CK(cudaMemcpyAsync(out_rgb + host_px * 3, d_rgb + dev_px * 3, n_px * 12, cudaMemcpyDeviceToHost, s));
    }
    if (out_rgb8 && n_px)
        CK(cudaMemcpyAsync(out_rgb8 + host_px * 3, static_cast<unsigned char*>(g.rgb8.p) + dev_px * 3, n_px * 3, cudaMemcpyDeviceToHost, s));
    if (out_mask && n_px) CK(cudaMemcpyAsync(out_mask + host_px, d_mask, n_px, cudaMemcpyDeviceToHost, s));
    float h_max = 0.f;
    if (stats) CK(cudaMemcpyAsync(&h_max, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(g.ev[3], s));
    CK(cudaStreamSynchronize(s));
    if (stats) {
        std::memset(stats, 0, sizeof(*stats));
        stats->max_value = (double)h_max;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[1], g.ev[2]));
        stats->ms_render = ms;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[3]));
        stats->ms_total = ms;
        stats->kernel_launches = launches;
        stats->resident_prims = resident;
        stats->d2h_bytes = (uint64_t)n_px * ((out_rgb ? 12 : 0) + (out_rgb8 ? 3 : 0) + (out_mask ? 1 : 0));
    }
    return RM_OK;
}

int rm_render_device(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id, void* d_max, void* stream) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!d_rgb || !d_max) return fail(RM_ERR_INVALID_ARGUMENT, "d_rgb and d_max must be device pointers");
    if (params && params->precision == RM_FP64)
        return render_device_impl<double>(scene, params, static_cast<double*>(d_rgb), d_prim_id, static_cast<double*>(d_max),
                                          static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, nullptr);
    return render_device_impl<float>(scene, params, static_cast<float*>(d_rgb), d_prim_id, static_cast<float*>(d_max),
                                     static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, nullptr);
}

int rm_render_device_rgb8(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id, void* d_max, uint8_t* d_rgb8,
                          void* stream) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!d_rgb || !d_max || !d_rgb8) return fail(RM_ERR_INVALID_ARGUMENT, "d_rgb, d_max and d_rgb8 must be device pointers");
    if (params && params->precision == RM_FP64)
        return render_device_impl<double>(scene, params, static_cast<double*>(d_rgb), d_prim_id, static_cast<double*>(d_max),
                                          static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, nullptr, nullptr, d_rgb8);
    return render_device_impl<float>(scene, params, static_cast<float*>(d_rgb), d_prim_id, static_cast<float*>(d_max),
                                     static_cast<cudaStream_t>(stream), 0, nullptr, nullptr, nullptr, nullptr, d_rgb8);
}

int rm_tonemap_device_busy(RmScene scene, const RmParams* params, const void* d_rgb, const void* d_max, int normalise,
                           uint8_t* d_rgb8, void* stream) {
    {
        std::lock_guard<std::mutex> lock(g.mu);
        if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
        int rc = check_params(params);
        if (rc != RM_OK) return rc;
        if (!d_rgb || !d_rgb8 || (normalise && !d_max)) return fail(RM_ERR_INVALID_ARGUMENT, "null device pointer");
        auto it = g.scenes.find(scene);
        if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
        const LastFrame& lf = it->second.last;
        auto fp = rm::make_frame_params<float>(*params);
        if (params->precision != RM_FP64 && lf.scheduled && lf.rgb8 == d_rgb8 && lf.width == fp.width && lf.height == fp.height &&
            lf.row_begin == fp.row_begin && lf.row_step == fp.row_step && lf.n_bands == fp.n_bands && lf.buf_row0 == 0) {
            CK(rm::launch_tonemap_busy(it->second.f32.ds, fp, static_cast<const float*>(d_rgb), static_cast<const float*>(d_max),
                                       normalise != 0, d_rgb8, static_cast<cudaStream_t>(stream)));
            return RM_OK;
        }
    }
    return rm_tonemap_device(params, d_rgb, d_max, normalise, d_rgb8, stream);      // no schedule to lean on: every tile
}

int rm_set_profiling(int on) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (on && g.prof.empty()) {
        g.prof.resize(kProfRing);
        for (auto& ps : g.prof)
            for (auto& ev : ps.e) CK(cudaEventCreate(&ev));
    }
    g.profiling = on != 0;
    g.prof_head = -1;
    g.prof_frames = 0;
    return RM_OK;
}

int rm_kernel_times(int back, double* ms_prepare, double* ms_render, double* ms_tonemap) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (back < 0 || back >= kProfRing || back >= g.prof_frames || g.prof_head < 0)
        return fail(RM_ERR_INVALID_ARGUMENT, "no such profiled frame: call rm_set_profiling(1) and render first (256 frames are kept)");
    const ProfSlot& ps = g.prof[(g.prof_head - back + kProfRing) % kProfRing];
    CK(cudaEventSynchronize(ps.e[ps.has_tone ? 3 : 2]));
    float a = 0.f, b = 0.f, c = -1.f;
    if (ps.split) {
        CK(cudaEventElapsedTime(&a, ps.e[0], ps.e[1]));
        CK(cudaEventElapsedTime(&b, ps.e[1], ps.e[2]));
    } else {
        CK(cudaEventElapsedTime(&b, ps.e[0], ps.e[2]));        // K0 and K1 overlap: one figure for both
    }
    if (ps.has_tone) CK(cudaEventElapsedTime(&c, ps.e[2], ps.e[3]));
    if (ms_prepare) *ms_prepare = a;
    if (ms_render) *ms_render = b;
    if (ms_tonemap) *ms_tonemap = c;
    return RM_OK;
}

int rm_last_kernel_times(double* ms_prepare, double* ms_render) { return rm_kernel_times(0, ms_prepare, ms_render, nullptr); }

int rm_scene_accel_status(RmScene scene, int32_t out_words[16]) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    auto it = g.scenes.find(scene);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    if (!it->second.f32.ready || !it->second.f32.ds.bvh.status) return fail(RM_ERR_INVALID_ARGUMENT, "scene has no FP32 pack");
    CK(cudaDeviceSynchronize());
    int32_t w[16];
    CK(cudaMemcpy(w, it->second.f32.ds.bvh.status, sizeof w, cudaMemcpyDeviceToHost));
    if (out_words) std::memcpy(out_words, w, sizeof w);
    if (w[0]) return fail(RM_ERR_CUDA, "a walk of the scene's hierarchy exceeded its node budget (corrupt hierarchy memory?): the frame is not valid");
    return RM_OK;
}

int rm_scene_walk_stats(RmScene scene, uint64_t out[3], int reset) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    auto it = g.scenes.find(scene);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    if (!it->second.f32.ready || !it->second.f32.ds.bvh.status) return fail(RM_ERR_INVALID_ARGUMENT, "scene has no FP32 pack");
    CK(cudaDeviceSynchronize());
    unsigned long long v[3] = {0, 0, 0};
    CK(cudaMemcpy(v, it->second.f32.ds.bvh.status + 10, sizeof v, cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(it->second.f32.ds.bvh.status + 10, 0, sizeof v));
    if (out) for (int i = 0; i < 3; i++) out[i] = v[i];
    return RM_OK;
}

int rm_scene_query_count(RmScene scene, uint64_t* out_queries, int reset) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    auto it = g.scenes.find(scene);
    if (it == g.scenes.end()) return fail(RM_ERR_INVALID_ARGUMENT, "unknown scene handle");
    if (!it->second.f32.ready || !it->second.f32.ds.ctr) return fail(RM_ERR_INVALID_ARGUMENT, "scene has no FP32 pack");
    CK(cudaDeviceSynchronize());
    unsigned long long v = 0;
    CK(cudaMemcpy(&v, it->second.f32.ds.ctr + 6, sizeof v, cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(it->second.f32.ds.ctr + 6, 0, sizeof v));
    if (out_queries) *out_queries = v;
    return RM_OK;
}

// ---- one frame across the GPUs of a box (include/rm_b200.h) ---------------------------------------------------------

int rm_peer_alloc(size_t bytes, void** d_ptr, unsigned char handle[RM_IPC_HANDLE_BYTES]) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (!d_ptr || !bytes) return fail(RM_ERR_INVALID_ARGUMENT, "d_ptr is null or bytes is 0");
    static_assert(sizeof(cudaIpcMemHandle_t) == RM_IPC_HANDLE_BYTES, "RM_IPC_HANDLE_BYTES must equal sizeof(cudaIpcMemHandle_t)");
    void* p = nullptr;
    CK(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    if (e == cudaSuccess && handle) {
        cudaIpcMemHandle_t h;
        e = cudaIpcGetMemHandle(&h, p);
        if (e == cudaSuccess) std::memcpy(handle, &h, sizeof h);
    }
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail_cuda(e, "rm_peer_alloc");
    }
    *d_ptr = p;
    return RM_OK;
}

int rm_peer_open(const unsigned char handle[RM_IPC_HANDLE_BYTES], void** d_ptr) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (!handle || !d_ptr) return fail(RM_ERR_INVALID_ARGUMENT, "handle or d_ptr is null");
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    CK(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return RM_OK;
}

int rm_peer_close(void* d_ptr) {
    if (!d_ptr) return RM_OK;
    CK(cudaIpcCloseMemHandle(d_ptr));
    return RM_OK;
}

int rm_peer_free(void* d_ptr) {
    if (!d_ptr) return RM_OK;
    CK(cudaFree(d_ptr));
    return RM_OK;
}

int rm_render_frame(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id, void* d_max, const RmExchange* x,
                    uint32_t seq, int normalise, void* stream) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed): no CUDA device bound");
    if (!d_rgb || !d_max || !x) return fail(RM_ERR_INVALID_ARGUMENT, "d_rgb, d_max and exchange are required");
    if (params && params->precision != RM_FP32) return fail(RM_ERR_INVALID_ARGUMENT, "rm_render_frame computes in RM_FP32");
    if (x->world < 1 || x->world > RM_MAX_RANKS || x->rank < 0 || x->rank >= x->world)
        return fail(RM_ERR_INVALID_ARGUMENT, "exchange: need 0 <= rank < world <= RM_MAX_RANKS");
    if (seq == 0) return fail(RM_ERR_INVALID_ARGUMENT, "frame sequence numbers start at 1 (mailboxes are zero-initialised)");
    rm::PeerLink link;
    link.rank = x->rank;
    link.world = x->world;
    link.seq = seq;
    for (int r = 0; r < x->world; r++) {
        if (!x->mailbox[r]) return fail(RM_ERR_INVALID_ARGUMENT, "exchange: mailbox pointer of a rank is null");
        link.box[r] = static_cast<unsigned long long*>(x->mailbox[r]);
    }
    unsigned char* frame8 = x->frame8[seq & 1u];
    unsigned char* frame8_next = x->frame8[(seq + 1u) & 1u];
    if (!frame8 || (x->rank == 0 && x->world > 1 && !frame8_next)) return fail(RM_ERR_INVALID_ARGUMENT, "exchange: frame8[] is null");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    rm::FrameParams<float> fp;
    // K0 + K1; K1 ends with the exchange and the conversion to 8 bits (K4 fused).  Only rank 0 clears bytes of the 8-bit
    // frames (its own black pixels in this frame's buffer, the whole bands of the other ranks in the next frame's buffer):
    // zeros never travel over NVLink.
    int rc = render_device_impl<float>(scene, params, static_cast<float*>(d_rgb), d_prim_id, static_cast<float*>(d_max), s, 0,
                                       nullptr, &fp, nullptr, nullptr, x->rank == 0 ? frame8 : nullptr, nullptr, &link, frame8,
                                       normalise != 0, frame8_next, true);
    if (rc != RM_OK) return rc;
    auto it = g.scenes.find(scene);
    const rm::DeviceScene<float>& ds = it->second.f32.ds;
    if (fp.n_bands <= 0) {
        // a rank without bands (more ranks than patch rows) still owes the others its word -- a maximum of zero -- and
        // rank 0 its signal (on rank 0: still has to wait for everybody else)
        CK(rm::launch_publish_zero(link, static_cast<float*>(d_max), s));
        CK(rm::launch_tonemap_peer(ds, fp, static_cast<const float*>(d_rgb), static_cast<const float*>(d_max), normalise != 0, frame8, s, link));
    }
    if (g.profiling && g.prof_head >= 0) {
        ProfSlot& ps = g.prof[g.prof_head];
        if (fp.n_bands <= 0) {                                  // nothing rendered: K0 and K1 take no time
            CK(cudaEventRecord(ps.e[0], s));
            CK(cudaEventRecord(ps.e[2], s));
        }
        ps.has_tone = false;                                    // K4 is part of K1 on this path
    }
    return RM_OK;
}

long long rm_graph_launch_count(void) { return g.graph_launches; }

int rm_peer_stamps(const RmExchange* x, uint64_t out_ns[7]) {
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (!x || !out_ns || x->rank < 0 || x->rank >= RM_MAX_RANKS || !x->mailbox[x->rank]) return fail(RM_ERR_INVALID_ARGUMENT, "exchange, out_ns or own mailbox is null");
    CK(cudaMemcpy(out_ns, static_cast<const unsigned long long*>(x->mailbox[x->rank]) + 56, 7 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return RM_OK;
}

int rm_peer_status(const RmExchange* x) {
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    if (!x || x->rank < 0 || x->rank >= RM_MAX_RANKS || !x->mailbox[x->rank]) return fail(RM_ERR_INVALID_ARGUMENT, "exchange or own mailbox is null");
    unsigned long long w = 0;
    CK(cudaMemcpy(&w, static_cast<const unsigned long long*>(x->mailbox[x->rank]) + 48, sizeof w, cudaMemcpyDeviceToHost));
    if (w) {
        char buf[160];
        std::snprintf(buf, sizeof buf, "a rank of the box did not answer within 2 s during the exchange of frame %u", (unsigned)(w >> 32));
        return fail(RM_ERR_PEER, buf);
    }
    return RM_OK;
}

int rm_render_device_stats(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id, void* d_max, void* stream,
                           RmStats* stats) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!d_rgb || !d_max || !stats) return fail(RM_ERR_INVALID_ARGUMENT, "d_rgb, d_max and stats are required");
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    int rc;
    if ((rc = g.small.ensure(1024)) != RM_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(static_cast<char*>(g.small.p) + 64);
    CK(cudaMemsetAsync(d_cnt, 0, rm::C_COUNT * 8, s));
    int resident = 0;
    if (params && params->precision == RM_FP64)
        rc = render_device_impl<double>(scene, params, static_cast<double*>(d_rgb), d_prim_id, static_cast<double*>(d_max), s, 0,
                                        d_cnt, nullptr, &resident);
    else
        rc = render_device_impl<float>(scene, params, static_cast<float*>(d_rgb), d_prim_id, static_cast<float*>(d_max), s, 0,
                                       d_cnt, nullptr, &resident);
    if (rc != RM_OK) return rc;
    unsigned long long host[rm::C_COUNT];
    CK(cudaMemcpyAsync(host, d_cnt, sizeof host, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::memset(stats, 0, sizeof(*stats));
    fill_counters(stats, host);
    stats->kernel_launches = 1;
    stats->resident_prims = resident;
    return RM_OK;
}

int rm_tonemap_device(const RmParams* params, const void* d_rgb, const void* d_max, int normalise, uint8_t* d_rgb8, void* stream) {
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    int rc = check_params(params);
    if (rc != RM_OK) return rc;
    if (!d_rgb || !d_rgb8 || (normalise && !d_max)) return fail(RM_ERR_INVALID_ARGUMENT, "null device pointer");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (params->precision == RM_FP64) {
        auto fp = rm::make_frame_params<double>(*params);
        CK(rm::launch_tonemap<double>(fp, static_cast<const double*>(d_rgb), static_cast<const double*>(d_max), normalise != 0, d_rgb8, s));
    } else {
        auto fp = rm::make_frame_params<float>(*params);
        CK(rm::launch_tonemap<float>(fp, static_cast<const float*>(d_rgb), static_cast<const float*>(d_max), normalise != 0, d_rgb8, s));
    }
    return RM_OK;
}

uint64_t rm_content_hash(const void* data, size_t bytes, uint64_t seed) { return data || !bytes ? hash_bytes(data, bytes, seed) : 0; }

void* rm_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void rm_host_free(void* p) { if (p) cudaFreeHost(p); }
int rm_host_register(void* p, size_t bytes) {
    CK(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
    return RM_OK;
}
int rm_host_unregister(void* p) {
    CK(cudaHostUnregister(p));
    return RM_OK;
}

int rm_measure_fp32_peak(double* out_tflops, double* out_ms) {
    std::lock_guard<std::mutex> lock(g.mu);
    if (!g.ready) return fail(RM_ERR_NOT_INITIALISED, "rm_init() has not been called (or failed)");
    const int blocks = g.prop.multiProcessorCount * 8;
    const int iters = 1 << 15;
    int rc;
    if ((rc = g.rgb.ensure((size_t)blocks * 256 * sizeof(float))) != RM_OK) return rc;
    double flops = 0;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {          // first repetition warms up
        CK(cudaEventRecord(g.ev[0], g.stream));
        CK(rm::launch_ffma_probe(static_cast<float*>(g.rgb.p), iters, blocks, g.stream, &flops));
        CK(cudaEventRecord(g.ev[1], g.stream));
        CK(cudaStreamSynchronize(g.stream));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev[0], g.ev[1]));
        if (rep > 0 && ms < best) best = ms;
    }
    if (out_ms) *out_ms = best;
    if (out_tflops) *out_tflops = flops / (best * 1e-3) / 1e12;
    return RM_OK;
}

}  // extern "C"
