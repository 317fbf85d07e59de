/*
 * rm_b200.h -- C ABI of the B200-native render hot path of rusty-marcher.
 *
 * This is the drop-in boundary.  In the reference the whole hot path sits inside
 *     Renderer::render(&self, frame: &mut FrameBuffer, scene: &Scene) -> String
 * (engine/src/renderer.rs:36-126): a Rayon `into_par_iter` over 32x32 pixel patches
 * (renderer.rs:63-89) followed by a single-threaded reassembly copy (renderer.rs:92-108).
 * A maintainer replaces exactly those lines with one call to rm_render(); everything the
 * kernels need is passed as plain f64 PODs that mirror the reference's own structs field
 * by field (the reference computes in f64, engine/src/geometry.rs:4-8).  No torch, CUDA or
 * C++ types appear in any signature.  INTEGRATION.md shows the Rust `extern "C"` block,
 * build.rs and the `Shape::flatten` glue.
 *
 * Error convention: every int-returning call yields RM_OK (0) or a negative RmStatus;
 * rm_last_error() returns the message of the last failure on the calling thread.  There
 * is NO CPU fallback: without a usable sm_100 device rm_init() fails with RM_ERR_NO_DEVICE
 * and every other entry point with RM_ERR_NOT_INITIALISED.
 */
#ifndef RM_B200_H
#define RM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RM_ABI_VERSION 5

typedef enum RmStatus {
    RM_OK = 0,
    RM_ERR_NO_DEVICE = -1,        /* no CUDA device / not an sm_100 part / driver error at init      */
    RM_ERR_NOT_INITIALISED = -2,
    RM_ERR_INVALID_ARGUMENT = -3, /* null pointer, bad handle, negative count ...                     */
    RM_ERR_DIMENSIONS = -4,       /* width not a multiple of the patch size (renderer.rs:107 panics)  */
    RM_ERR_SCENE = -5,            /* malformed flat scene (index out of range, polygon with <3 verts) */
    RM_ERR_CUDA = -6,             /* a CUDA runtime call failed; see rm_last_error()                  */
    RM_ERR_OUT_OF_MEMORY = -7,
    RM_ERR_PEER = -8              /* a rank of the box did not answer within 2 s during a frame's exchange */
} RmStatus;

/* ---- scene PODs: field-for-field mirrors of the reference structs (all f64) ------------------ */

/* engine/src/shapes.rs:21-32  struct Reflectance */
typedef struct RmReflectance {
    double  diffusion;
    double  diffuse_color[3];
    double  specular;
    double  specular_exponent;
    int32_t is_glass_like;
    double  reflection;
    double  refractive_index;
} RmReflectance;

/* engine/src/sphere.rs:6-11  struct Sphere (bounding_box is dead on the hot path) */
typedef struct RmSphere {
    double        center[3];
    double        radius_square;
    RmReflectance reflectance;
} RmSphere;

/* engine/src/polygon.rs:6-12  struct ConvexPolygon; vertices live in RmFlatScene.polygon_vertices */
typedef struct RmPolygon {
    int32_t       first_vertex;
    int32_t       n_vertices;
    double        plane_normal[3];
    double        plane_point[3];
    RmReflectance reflectance;
} RmPolygon;

/* engine/src/triangle.rs:6-10  struct Triangle (vertices, precomputed normal and center) */
typedef struct RmTriangle {
    double vertices[9];
    double normal[3];
    double center[3];
} RmTriangle;

/* engine/src/obj.rs:14-20  struct Obj: a run of triangles + their per-triangle reflectances */
typedef struct RmObj {
    int32_t first_triangle;
    int32_t n_triangles;
} RmObj;

/* engine/src/lights.rs:4-8  struct Light (color already L-inf normalised by create_light) */
typedef struct RmLight {
    double position[3];
    double color[3];
    double intensity;
} RmLight;

typedef enum RmShapeKind { RM_SHAPE_SPHERE = 0, RM_SHAPE_POLYGON = 1, RM_SHAPE_OBJ = 2 } RmShapeKind;

/* one entry of Scene.shapes (engine/src/scene.rs:11), in scene order */
typedef struct RmShapeRef {
    int32_t kind;    /* RmShapeKind */
    int32_t index;   /* into spheres / polygons / objs */
} RmShapeRef;

/* engine/src/scene.rs:9-13  struct Scene, flattened.  All arrays are host memory owned by the
 * caller and are copied by rm_scene_upload().  The primitive id reported by rm_render is the index
 * in the list obtained by walking `shapes` in order, an Obj counting once per triangle. */
typedef struct RmFlatScene {
    int32_t              n_shapes;
    const RmShapeRef*    shapes;
    int32_t              n_spheres;
    const RmSphere*      spheres;
    int32_t              n_polygons;
    const RmPolygon*     polygons;
    int32_t              n_polygon_vertices;
    const double*        polygon_vertices;        /* xyz triples */
    int32_t              n_objs;
    const RmObj*         objs;
    int32_t              n_triangles;
    const RmTriangle*    triangles;
    const RmReflectance* triangle_reflectances;   /* n_triangles entries (obj.rs:17) */
    int32_t              n_lights;
    const RmLight*       lights;
} RmFlatScene;

typedef enum RmPrecision {
    RM_FP32 = 0,   /* production kernels: FP32 CUDA cores                                          */
    RM_FP64 = 1    /* validation kernels: the reference's f64 arithmetic, operation for operation */
} RmPrecision;

/* Per-frame parameters.  rm_params_default() fills in the constants the reference hard-codes. */
typedef struct RmParams {
    int32_t width;            /* FrameBuffer.width  (framebuffer.rs:7); multiple of patch_size      */
    int32_t height;           /* FrameBuffer.height (framebuffer.rs:8)                              */
    double  fov;              /* create_renderer(fov, ..) radians (renderer.rs:25, main.rs:368: 1.5)*/
    double  camera[3];        /* Scene.camera (scene.rs:12)                                         */
    int32_t max_depth;        /* cast_ray depth cap, renderer.rs:262: 3                             */
    double  background;       /* renderer.rs:40-44: 0.1                                             */
    int32_t patch_size;       /* renderer.rs:47: 32 (only 32 is supported)                          */
    int32_t precision;        /* RmPrecision                                                        */
    int32_t patch_row_begin;  /* row tile of this call, in patch rows; [0, -1) = every rendered row */
    int32_t patch_row_end;
    int32_t cull_backfacing;  /* drop planar primitives that can never pass the reference's z-only
                                 inside test (projected winding not CCW); 0 = keep all             */
    int32_t patch_row_stride; /* render patch rows begin, begin + stride, ... < end (0 and 1 = every
                                 row).  Rank k of G renders rows k, k + G, ...: interleaved row tiles
                                 balance scenes whose work sits in one part of the frame           */
    int32_t accel;            /* 0 = every scene query tests every resident primitive, the reference's
                                 traversal (shapes.rs:92-143, obj.rs:186-216); 1 = queries walk a bounding-
                                 volume hierarchy over the hittable primitives (the bounding boxes the
                                 reference carries but never uses, shapes.rs:34-38,63-86).  Same tests per
                                 (ray, primitive), same winner: the FP32 frame is bit-identical, the work per
                                 segment drops from O(n) to O(log n).  RM_FP32 production kernel only.
                                 2 = the same through the instantiation that also counts its work (node visits,
                                 leaf tests: rm_scene_walk_stats) -- for measurement, a few percent slower       */
} RmParams;

/* Event counters (same definitions as SURVEY.md 8d) + timings of one call. */
typedef struct RmStats {
    uint64_t pixels, closest_segments, anyhit_segments;
    uint64_t sphere_tests, sphere_disc, sphere_hits;
    uint64_t plane_tests, plane_dist, plane_point, edge_tests;
    uint64_t cand_dist, hits, light_evals, lit_lights;
    uint64_t glass_hits, reflections, refractions;
    double   max_value;       /* FrameBuffer::normalize's max (framebuffer.rs:59-69) over rendered rows */
    double   ms_render;       /* device time of the render kernel(s), CUDA events                       */
    double   ms_total;        /* device time of the whole call incl. copies                             */
    int32_t  kernel_launches; /* kernels launched by this call                                          */
    int32_t  resident_prims;  /* primitives actually traced (after culling)                             */
    uint64_t d2h_bytes;       /* bytes this call copied from device to host memory                      */
} RmStats;

typedef int64_t RmScene;   /* opaque handle, > 0 */

/* ---- lifecycle --------------------------------------------------------------------------------- */
int         rm_abi_version(void);
int         rm_init(int device);            /* binds the calling process to CUDA device `device` */
void        rm_shutdown(void);
const char* rm_last_error(void);
int         rm_device_info(char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz);
void        rm_params_default(RmParams* p, int width, int height);
void        rm_reflectance_default(RmReflectance* r);     /* shapes.rs:50-60 */

/* ---- scene ------------------------------------------------------------------------------------- */
int rm_scene_upload(const RmFlatScene* scene, RmScene* out_handle);
int rm_scene_free(RmScene handle);
int rm_scene_num_prims(RmScene handle);

/* ---- the hot path, host buffers (what Renderer::render binds) -------------------------------- *
 * Renders patch rows [patch_row_begin, patch_row_end) and copies the results to HOST memory.
 *   out_rgb     H*W*3 floats (RM_FP32) row-major RGB, or NULL.  Only rendered rows are written;
 *               the rest of the buffer is left untouched like frame.buffer in the reference.
 *   out_prim_id H*W int32: primitive hit by the primary ray, -1 = miss; or NULL.
 *   out_rgb8    H*W*3 bytes: normalize() + to_vec() of the rendered tile (framebuffer.rs:40-82),
 *               normalised by this call's own max; or NULL.
 *   stats       optional; counters are only collected when stats->pixels is set to 1 on entry
 *               (instrumented kernel, slower), timings always.
 * Host buffers may be pageable; pinned ones (rm_host_alloc / rm_host_register) copy faster. */
int rm_render(RmScene scene, const RmParams* params, float* out_rgb, int32_t* out_prim_id,
              uint8_t* out_rgb8, RmStats* stats);
/* rm_render with only out_rgb given (the float frame, what Renderer::render returns) delivers through the packed path
 * described at rm_render_rows_f64 below; the rows it writes are bit-identical. */
/* Same with RM_FP64 arithmetic and a double framebuffer (validation mode). */
int rm_render_f64(RmScene scene, const RmParams* params, double* out_rgb, int32_t* out_prim_id,
                  uint8_t* out_rgb8, RmStats* stats);

/* ---- the hot path into the reference's own frame type ------------------------------------------------------------------ *
 * FrameBuffer.buffer is a Vec<Vec<Vec3f>> (engine/src/framebuffer.rs:6-10): one heap allocation per pixel row, f64
 * channels.  rows[y] (y < params->height) points to row y: width * 3 doubles (rm_render_rows_f64; the FP32 results widened,
 * exactly) or floats (rm_render_rows_f32).  Only rows of the call's bands are touched, like renderer.rs:92-108.
 * Delivery: when the frame has a tile schedule (triangle-only scenes) only the busy tiles cross PCIe.  Into a contiguous
 * float32 frame in pinned host memory (rm_host_alloc / rm_host_register; rm_render with out_rgb only, rm_render_rows_f32
 * with rows that follow each other) the device writes them itself, tile row by tile row (RM_B200_DIRECT_DELIVERY=0: never);
 * otherwise they are packed on the device, cross in a few chunked copies into a staging buffer and are scattered / widened
 * by the library's host threads (RM_B200_HOST_THREADS, default: all).  Either way those threads zero-fill the provably
 * black tiles meanwhile -- from the moment the prepare kernel's schedule is on the host, while the frame is still being
 * rendered (RM_B200_EARLY_SCHEDULE=0: only once the render kernel is done).
 * flags: RM_ROWS_RETAINED -- the caller has not touched the frame since the library's previous delivery into it (the
 * re-render loop of engine/src/main.rs:329-351 keeps one FrameBuffer): only tiles that held something then and are black
 * now are cleared.  The first delivery into a frame clears every black tile regardless.  stats: timings, max_value.
 * RM_FP32 only. */
#define RM_ROWS_RETAINED 1
int rm_render_rows_f64(RmScene scene, const RmParams* params, double* const* rows, int flags, RmStats* stats);
int rm_render_rows_f32(RmScene scene, const RmParams* params, float* const* rows, int flags, RmStats* stats);

/* ---- extension mode: per-channel refractive indices (BASELINE.json configs[3]; SURVEY.md 8d item 4) ---------- *
 * The reference has ONE scalar refractive index per material (shapes.rs:21-32, optics.rs:8-89); there is no reference
 * behaviour for dispersion.  Defined here -- and identically in the oracle (oracle.render_dispersive) -- as three passes
 * of the unchanged hot path: scenes[c] is the scene with every glass-like material at the index of channel c
 * (c = 0, 1, 2 for R, G, B; the caller uploads the three variants, geometry and lights identical), and channel c of the
 * frame is channel c of pass c.  out_prim_id: the primary ids (they do not depend on the index).  stats: timings,
 * launches; max_value is not computed (FrameBuffer::normalize computes it from the frame, framebuffer.rs:58-69).
 * RM_FP32, contiguous patch rows (patch_row_stride <= 1). */
int rm_render_dispersive(const RmScene scenes[3], const RmParams* params, float* out_rgb, int32_t* out_prim_id,
                         RmStats* stats);

/* ---- extension mode: supersampled anti-aliasing, s x s samples per pixel -------------------------------------------------- *
 * The reference traces one primary ray per pixel (renderer.rs:63-89); there is no reference behaviour for anti-aliasing.
 * Defined here -- and identically in the tests' f64 restatement over the oracle -- in terms of the FP32 production render:
 * for samples = s in [1, 8], pixel (x, y) of the frame is the mean of the FP32 render of the same scene and camera at width
 * s*W and height s*H over the s x s block of sub-pixels (s*x + j, s*y + i), i, j in [0, s).  backproject (renderer.rs:128-135)
 * divides by the width, so the sub-pixel rays are the reference's rays at x + j/s; the aspect ratio (s*W)/(s*H) rounds to the
 * same double as W/H.  The mean is FP32 in this order (normative; no fused multiply-add):
 *     acc = 0.f;  for i in [0, s): for j in [0, s): acc += v[i][j];  out = acc / (float)(s*s)      (IEEE division)
 * Rows: the output patch rows [b, e) of the call (patch_row_end = -1: floor(H/32)), like rm_render; the s x frame renders
 * exactly its patch rows [s*b, s*e) -- not floor(s*H/32) bands.  Other rows of the caller's buffers are left untouched.
 *   out_rgb   H*W*3 floats, or NULL: the resolved frame.
 *   out_rgb8  H*W*3 bytes, or NULL: normalize() + to_vec() of the resolved rows by their own maximum (framebuffer.rs:40-82).
 *             At least one of the two must be given.
 *   stats     optional: max_value (FrameBuffer::normalize's max over the resolved rows), ms_render (device time of the s x
 *             frame's render kernels), ms_total, kernel_launches (the resolve included), resident_prims, d2h_bytes.  Event
 *             counters are not collected.
 * s = 1 gives rm_render's frame bit for bit.  accel and cull_backfacing apply to the s x render.  Device memory: a scratch of
 * 12 * s^2 * W * rows bytes for the s x frame (rows = rendered pixel rows; 1.6 GB for a 3840 x 2160 frame at s = 4), kept for
 * the next call.  The call writes the caller's float frame, so the library forgets its previous deliveries into that memory
 * (RM_ROWS_RETAINED, above): the next retained delivery there clears every black tile.
 * RM_ERR_INVALID_ARGUMENT: samples outside [1, 8], precision other than RM_FP32, patch_row_stride > 1, unknown scene, both
 * outputs NULL.  RM_ERR_DIMENSIONS: the s x frame is not a valid frame (s*W or s*H above 65535, 2^22 patches or more). */
int rm_render_supersampled(RmScene scene, const RmParams* params, int samples, float* out_rgb, uint8_t* out_rgb8,
                           RmStats* stats);

/* ---- extension mode: adaptive anti-aliasing, s x s samples only where the frame changes abruptly ---------------------------- *
 * Whitted's (1980) adaptive supersampling with Mitchell's (1987) contrast test; no reference behaviour.  Defined by two calls:
 * P = rm_render's FP32 frame of the scene and camera with its primary ids, S = rm_render_supersampled(..., samples)'s frame.
 * With R = 32 * floor(H/32) (the rendered rows), pixel p = (x, y) is REFINED if contrast < 0 (every pixel), or else if one of
 * its 8 neighbours q inside [0, W) x [0, R) has id(q) != id(p), or, for some channel c with a = P[p][c], b = P[q][c],
 *     fabsf(a - b) > k * (a + b),     k = (float)contrast, every operation rounded to FP32, no fused multiply-add.
 * contrast = +inf refines geometric edges only (inf * 0 is NaN, the comparison false).  The output pixel is S[p] if p is
 * refined, P[p] otherwise: samples = 1 gives rm_render's frame, contrast < 0 rm_render_supersampled's, and every other frame
 * follows bit for bit from those two and the mask.  Sub-pixel detail wholly inside one pixel (a thin object that no pixel
 * centre hits, a highlight between two samples) changes no 1x pixel and is missed by design.
 * Rows: the output patch rows [b, e) of the call (patch_row_end = -1: floor(H/32)), like rm_render; rows outside are left
 * untouched in all three outputs.  The mask looks at neighbours outside the call's rows as well (the 1x frame is rendered
 * over one more patch row on either side), so a call over some patch rows gives the same rows as a full-frame call.
 *   out_rgb   H*W*3 floats, or NULL: the frame.
 *   out_rgb8  H*W*3 bytes, or NULL: normalize() + to_vec() of the output rows by their own maximum.  At least one of the two.
 *   out_mask  H*W bytes, or NULL: 1 = refined, 0 = not.
 *   stats     optional: max_value (over the output rows), ms_render (device time from the start of the 1x render to the
 *             resolved float rows: no tone map, no copies), ms_total, kernel_launches, resident_prims, d2h_bytes.
 * Device memory, kept for the next call: the 1x frame's rows (16 W bytes per row, halo included), W * rows * 5 bytes for the
 * mask and the list of refined pixels, and the refined pixels' sub-pixel values, sized for the worst case (every pixel
 * refined): 12 * s^2 * W * rows bytes, as rm_render_supersampled's scratch (1.6 GB for a 3840 x 2160 frame at s = 4).
 * The call writes the caller's float frame, so the library forgets its previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: samples outside [1, 8], NaN contrast, precision other than RM_FP32, patch_row_stride > 1,
 * max_depth < 1, unknown scene, out_rgb and out_rgb8 both NULL.  RM_ERR_DIMENSIONS: the s x frame is not a valid frame (as for
 * rm_render_supersampled). */
int rm_render_adaptive(RmScene scene, const RmParams* params, int samples, double contrast, float* out_rgb, uint8_t* out_rgb8,
                       uint8_t* out_mask, RmStats* stats);

/* ---- the hot path, device buffers (no copies; for callers that keep frames in HBM) ----------- *
 * d_rgb: device float (RM_FP32) or double (RM_FP64) H*W*3; d_prim_id optional; d_max: device
 * scalar of the same type as d_rgb that receives max(previous value, tile max) -- zero it first.
 * `stream` is a cudaStream_t (NULL = default stream).  Asynchronous. */
int rm_render_device(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id,
                     void* d_max, void* stream);
/* rm_render_device that also prepares the 8-bit frame d_rgb8 (H*W*3 bytes, may be a peer-mapped pointer of another
 * GPU): when the frame can be rendered with a tile schedule (triangle-only scenes) the render kernel zeroes the bytes
 * of every pixel it visits -- quantize(0 * 1/max) is 0 whatever the maximum (framebuffer.rs:71-82) -- and
 * rm_tonemap_device_busy() then only converts the tiles that can hold anything else. */
int rm_render_device_rgb8(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id,
                          void* d_max, uint8_t* d_rgb8, void* stream);
/* rm_tonemap_device for the frame `scene` rendered last through rm_render_device_rgb8 with the same params and
 * d_rgb8; converts only the busy tiles when that render had a tile schedule, every tile otherwise. */
int rm_tonemap_device_busy(RmScene scene, const RmParams* params, const void* d_rgb, const void* d_max,
                           int normalise, uint8_t* d_rgb8, void* stream);
/* Instrumented variant of rm_render_device: also accumulates the event counters (synchronous). */
int rm_render_device_stats(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id,
                           void* d_max, void* stream, RmStats* stats);
/* FrameBuffer::normalize + to_vec on device (framebuffer.rs:40-82) for rows of this tile:
 * d_rgb8[y][x][c] = (u8)(255*clamp(d_rgb*(1/max),0,1)); d_rgb8 may be a peer-mapped pointer of
 * another GPU (fused gather).  normalise=0 gives the un-normalised display path (main.rs:337). */
int rm_tonemap_device(const RmParams* params, const void* d_rgb, const void* d_max, int normalise,
                      uint8_t* d_rgb8, void* stream);

/* 64-bit content hash of a byte range, at memory speed: the function the library keys its cache of packed scenes with
 * (a scene uploaded again with the same content is not packed again).  Exported for bindings that keep caches of their own
 * keyed by content -- the Python mirror's scene fingerprint.  Needs no GPU. */
uint64_t rm_content_hash(const void* data, size_t bytes, uint64_t seed);

/* ---- pinned host memory helpers ---------------------------------------------------------------- */
void* rm_host_alloc(size_t bytes);
void  rm_host_free(void* p);
int   rm_host_register(void* p, size_t bytes);
int   rm_host_unregister(void* p);

/* ---- one frame on the GPUs of one box: render + the path's single exchange step, in two launches ---------- *
 * The reference's Rayon loop splits the frame into independent 32x32 patches (renderer.rs:46-89); across GPUs the
 * frame is split into 32-row bands (RmParams.patch_row_begin/end/stride; a rank renders every G-th band, from a first band of its own), one
 * process per GPU.  The only data the ranks must exchange is what FrameBuffer::normalize (framebuffer.rs:58-76) needs
 * -- ONE float, the global channel maximum -- and the finished 8-bit rows, which go to rank 0.  Both travel over
 * NVLink peer memory from inside the render kernel (no NCCL call on the path, two launches per frame and rank):
 *   K0  per-frame triangle records + tile schedule; zeroes d_max
 *   K1  renders this rank's bands (float rows stay local); rank 0 also clears the bytes of its own provably black pixels
 *       in the 8-bit frame.  The last CTA to retire from rendering stores {seq, max} into every rank's mailbox.  Then every
 *       CTA waits for the G mailbox words of frame `seq` (which doubles as the grid-wide barrier of this persistent
 *       kernel), takes their maximum, quantises this rank's busy tiles (normalize + to_vec, framebuffer.rs:40-82) straight
 *       into rank 0's 8-bit frame, and the last CTA signals rank 0.  While the tiles of the other ranks arrive, rank 0
 *       clears those ranks' bands in the OTHER 8-bit buffer, the one the next frame will use (local HBM stores: zeros
 *       never cross NVLink); its kernel retires only when all G ranks have signalled, so whatever follows it on rank 0's
 *       stream sees the complete frame.
 * Memory shared between the processes is allocated with rm_peer_alloc (cudaMalloc + CUDA IPC handle), the 64-byte
 * handle is passed to the other ranks by any means (torch.distributed / MPI / a pipe) and mapped with rm_peer_open.
 * world == 1 needs no peers: mailbox[0] and frame8[] are local allocations. */
#define RM_MAX_RANKS 16
#define RM_IPC_HANDLE_BYTES 64
#define RM_MAILBOX_BYTES 512
typedef struct RmExchange {
    int32_t  rank, world;
    void*    mailbox[RM_MAX_RANKS];  /* mailbox[r]: rank r's mailbox (RM_MAILBOX_BYTES, zeroed once), mapped on this GPU */
    uint8_t* frame8[2];              /* rank 0's 8-bit frames (H*W*3 bytes each, zeroed once by rm_peer_alloc); frame `seq` goes
                                        to frame8[seq & 1] and is valid until the next rm_render_frame is issued on rank 0's
                                        stream (that launch prepares the buffer for the frame after it)                  */
} RmExchange;
int rm_peer_alloc(size_t bytes, void** d_ptr, unsigned char handle[RM_IPC_HANDLE_BYTES]);  /* zero-filled */
int rm_peer_open(const unsigned char handle[RM_IPC_HANDLE_BYTES], void** d_ptr);
int rm_peer_close(void* d_ptr);                                                           /* of rm_peer_open  */
int rm_peer_free(void* d_ptr);                                                            /* of rm_peer_alloc */
/* Sharing the device.  K1 is a persistent kernel whose last phase waits, inside the kernel, until all of its CTAs have
 * finished rendering: every CTA of the grid must be resident.  The grid is sized for that on a GPU the calling process has
 * to itself.  If other work occupies SMs for long (another process under MPS, a long kernel of the caller on a second
 * stream), set RM_B200_COOPERATIVE=1: the launch then carries the cooperative attribute and the driver guarantees
 * co-residency (+2 to 3 us per frame).  A wait that is not answered within 2 s gives up, the frame is NOT valid and
 * rm_peer_status() reports RM_ERR_PEER -- check it after synchronising when frames matter.
 * One scene, one frame at a time: a scene's device pack holds the per-frame schedule and raster records, so renders of the
 * same scene are ordered by the library even across streams (a render issued on another stream waits for the previous one);
 * different scenes render concurrently. */
/* One frame (FP32).  d_rgb: this rank's float frame (H*W*3, rows of other ranks are not touched); d_max: device float,
 * receives this rank's maximum; seq >= 1 and equal on all ranks, incremented by one per frame.  Asynchronous on
 * `stream`.  After a synchronisation rm_peer_status() tells whether any wait on this GPU timed out (RM_ERR_PEER). */
int rm_render_frame(RmScene scene, const RmParams* params, void* d_rgb, int32_t* d_prim_id, void* d_max,
                    const RmExchange* exchange, uint32_t seq, int normalise, void* stream);
int rm_peer_status(const RmExchange* exchange);
/* Frames this process has issued as ONE CUDA graph launch.  With RM_B200_GRAPH=1 in the environment (read per call)
 * rm_render_frame, from a scene's second frame on, captures its kernel pair on a stream of the library's own, updates the
 * instantiated graph with the frame's parameters and launches it on the caller's stream.  Opt-in: on the device it measures
 * within +-0.6 us of the two plain launches (whose programmatic edge already overlaps K1's launch with K0); it saves 10 us
 * of HOST time per frame (40 instead of 51 us to issue one). */
long long rm_graph_launch_count(void);
/* %globaltimer stamps (ns) the render kernel left in this rank's mailbox during its last frame: [0] kernel start,
 * [1] rendering done (last CTA), [2] all ranks' maxima gathered, [3] this rank's 8-bit tiles stored, [4] rank 0 only:
 * every rank has signalled, frame complete, [5] / [6] start and end of the frame's prepare kernel (K0; 0 when the scene has
 * no tile schedule).  Synchronous (a small device-to-host copy); for phase breakdowns. */
int rm_peer_stamps(const RmExchange* exchange, uint64_t out_ns[7]);

/* ---- per-kernel device times (CUDA events on the launching stream around K0 and K1) ------------ *
 * rm_set_profiling(1) makes every following device render record three events; rm_last_kernel_times() waits for the
 * last one and returns the prepare (K0) and render (K1) kernel durations of that frame in milliseconds. */
int rm_set_profiling(int on);
int rm_last_kernel_times(double* ms_prepare, double* ms_render);
/* The same for the frame `back` frames before the last one (a ring of 256 frames is kept).  On the rm_render_frame path
 * K1 is launched programmatically dependent on K0 (its prologue overlaps K0) and ends with the exchange and the fused
 * K4: there ms_prepare is 0 and ms_render covers K0 + K1 + exchange + K4, ms_tonemap is -1.  On the other paths the
 * tone-map kernel is a separate call that is not timed here (ms_tonemap -1). */
int rm_kernel_times(int back, double* ms_prepare, double* ms_render, double* ms_tonemap);
/* Scene queries behind the primary rays -- closest-hit calls of the reflect/refract recursion (renderer.rs:266 at
 * level > 1) plus shadow rays (renderer.rs:174) -- issued by the accel = 1 renders of `scene` since the last reset.
 * Ray segments of a frame = rendered pixels + this count: the figure the instrumented brute-force kernel (RmStats)
 * gives for scenes small enough to run through it.  Synchronises the device. */
int rm_scene_query_count(RmScene scene, uint64_t* out_queries, int reset);
/* Work of the accel = 2 renders of `scene` since the last reset: out[0] node visits (one visit = the boxes of both
 * children: 64 bytes, two slab tests), out[1] sphere tests, out[2] plane tests (triangles and n-gons) at the leaves --
 * the algorithmic work of a frame rendered through the hierarchy (bench.py's roofline for accel workloads).
 * Synchronises the device. */
int rm_scene_walk_stats(RmScene scene, uint64_t out[3], int reset);
/* A walk of the hierarchy visits every node at most once; one that exceeds that budget (possible only with corrupt
 * hierarchy memory) gives up instead of hanging the GPU and raises a sticky flag.  Returns RM_OK while the flag is down,
 * RM_ERR_CUDA once it is up; out_words (optional): [0] flag, [1..6] origin and direction of the first such ray (float
 * bits), [7] node, [8] stack depth.  Synchronises the device. */
int rm_scene_accel_status(RmScene scene, int32_t out_words[16]);

/* ---- FP32 peak probe: a pure-FFMA kernel, returns measured TFLOP/s (roofline denominator) ----- */
int rm_measure_fp32_peak(double* out_tflops, double* out_ms);

#ifdef __cplusplus
}
#endif
#endif /* RM_B200_H */
