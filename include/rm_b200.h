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

/* ---- extension mode: camera orientation -- render from any view direction, not only down -z ------------------------------- *
 * The reference's camera looks down -z (backproject, renderer.rs:128-135); it has a position and a field of view only.
 * Definition (normative; the tests' f64 restatement over the oracle is the same):
 *   Basis, in f64 without fused multiply-add; normalized(a) = a.scale(1 / norm), norm = sqrt(x*x + y*y + z*z)
 *   (geometry.rs:104-109); cross(a, b) = (a.y*b.z - a.z*b.y, a.z*b.x - a.x*b.z, a.x*b.y - a.y*b.x):
 *       w = normalized(-forward);   u = normalized(cross(up, w));   v = cross(w, u)
 *   A view is invalid (RM_ERR_INVALID_ARGUMENT) if a component is not finite, if forward.forward == 0, or if
 *   |cross(up, w)|^2 <= 1e-20 * (up.up) -- up = 0 or parallel to forward.
 *   Primary rays: with (dx, dy, dz) the reference's normalised backproject direction of pixel (j, i), the primary ray leaves
 *   the camera position along
 *       d = ((u.x*dx + v.x*dy) + w.x*dz,  (u.y*dx + v.y*dy) + w.y*dz,  (u.z*dx + v.z*dy) + w.z*dz)
 *   without renormalisation.  Everything after the primary ray is the reference's: recursion, shading, lights.
 *   Identity: a view whose basis is exactly u = (1,0,0), v = (0,1,0), w = (0,0,1) (forward = (0,0,-1), up = (0,1,0) is one)
 *   is rendered by rm_render's own path: the frame, ids and 8-bit frame equal rm_render's bit for bit.
 *   Kept on purpose: the reference's triangle and polygon inside test looks at world z only (triangle.rs:13-15), so a turned
 *   camera still sees only planar primitives whose world normal has z > 0, and cull_backfacing (a world-space criterion) stays
 *   valid.  The scene is not rotated into camera space: that would change which primitives can be hit.
 * FP32 production path: K0 writes the raster records rotated by the transposed basis (in f64), stage A runs on them unchanged,
 * and the world direction of a primary ray (spheres, n-gons, the hierarchy walk, shading) is the FP32 basis applied to the
 * unit camera-space direction; frames meet the same FP32 parity criteria against the f64 definition as rm_render's.  With
 * accel = 2 a view call renders as accel = 1 (the hierarchy without its work counters).
 * Out of scope: views for rm_render_supersampled, rm_render_adaptive, rm_render_dispersive, rm_render_rows_* and
 * rm_render_frame; projections other than the reference's pinhole; an up vector that turns with the camera. */
typedef struct RmView {
    double forward[3];   /* direction the camera looks in (need not be unit length) */
    double up[3];        /* approximate up; only its component orthogonal to forward matters */
} RmView;
/* u, v, w of `view` into out_basis[0..2], [3..5], [6..8], or RM_ERR_INVALID_ARGUMENT.  Needs no GPU. */
int rm_view_basis(const RmView* view, double out_basis[9]);
/* rm_render from the camera turned to `view`: the same outputs, rows (patch_row_begin / end / stride), stats semantics and
 * counter collection (stats->pixels = 1).  RM_FP32.  The call writes the caller's float frame itself, so the library forgets
 * its previous deliveries into that memory (RM_ROWS_RETAINED).  RM_ERR_INVALID_ARGUMENT: a NULL or invalid view, a precision
 * other than RM_FP32, and whatever rm_render rejects. */
int rm_render_view(RmScene scene, const RmParams* params, const RmView* view, float* out_rgb, int32_t* out_prim_id,
                   uint8_t* out_rgb8, RmStats* stats);
/* The same with RM_FP64 arithmetic and a double frame (validation mode, like rm_render_f64); params->precision RM_FP64. */
int rm_render_view_f64(RmScene scene, const RmParams* params, const RmView* view, double* out_rgb, int32_t* out_prim_id,
                       uint8_t* out_rgb8, RmStats* stats);
/* rm_render_device from the camera turned to `view` (RM_FP32 or RM_FP64 by params->precision). */
int rm_render_view_device(RmScene scene, const RmParams* params, const RmView* view, void* d_rgb, int32_t* d_prim_id,
                          void* d_max, void* stream);

/* ---- extension mode: depth of field -- a thin-lens camera with an aperture and a focus distance ---------------------------- *
 * The reference's pinhole keeps every depth in focus; a thin lens blurs what lies off the plane in focus.
 * Definition (normative; rm::lens_offset / rm::lens_ray in rm_trace.cuh are this, and the tests' restatement over the
 * oracle is the same).  All in f64 without fused multiply-add.  s = samples; c the camera position; u, v, w the view's
 * basis (rm_view_basis), or the identity without a view.  For output pixel (x, y) and sample (i, j), i, j in [0, s):
 *   1. d = the reference's normalised backproject direction of sub-pixel (s x + j, s y + i) in the s W x s H frame
 *      (rm_render_supersampled's sub-pixel ray).
 *   2. Lens point: a = (i + j) mod s, b = j (the shift decorrelates lens strata from sub-pixel strata);
 *      p = (2 a + 1) / s - 1, q = (2 b + 1) / s - 1;  lx = p * sqrt(1 - (q*q) * 0.5),  ly = q * sqrt(1 - (p*p) * 0.5)
 *      (the elliptical grid-to-disc map: every point lies in the unit disc).
 *   3. aperture = 0: the ray is (c, world(d)), the pinhole ray.  Otherwise
 *        k = focus / (-d.z);  P = (d.x*k, d.y*k, d.z*k);  L = (aperture*lx, aperture*ly, 0);
 *        e = normalized(P - L)  (geometry.rs's scale(1 / norm));
 *        origin = c + ((u*L.x + v*L.y)), component by component in that order;  direction = world(e),
 *      with world(e) = ((u.x*e.x + v.x*e.y) + w.x*e.z, ...) as for rm_render_view, not renormalised.
 *   4. The sample's value is the reference's cast_ray from that ray (renderer.rs:254-309, levels 1..max_depth); everything
 *      after the ray is unchanged, the world-z inside test of planar primitives included.
 *   5. The pixel is the FP32 mean of its s^2 sample values in rm_render_supersampled's order (sub-rows i outer, j inner).
 * Consequences:
 *   - aperture = 0 without a view is rm_render_supersampled's frame bit for bit (the call is routed there); with s = 1 that
 *     is also rm_render's frame.
 *   - Points on the plane at distance `focus` (along the view axis) stay sharp: every sample of a pixel aims at the same P.
 *   - At s = 1 the only lens point is the centre, so the lens has no effect.
 *   - The lens pattern is the same for every pixel: out-of-focus objects show as s^2 overlapping copies, not as noise.  The
 *     frame is deterministic by design.
 * FP32 production path (lens_kernel): each sample ray is computed in f64 by rm::lens_ray and traced with the general FP32
 * closest-hit query from level 1 on (brute force, or the hierarchy with accel != 0; accel = 2 renders as accel = 1), the rest
 * as rm_render's shading stage; frames meet the FP32 parity criteria against the f64 definition.  cull_backfacing applies.
 * Rows, outputs and stats as rm_render_supersampled: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched;
 * out_rgb (H*W*3 floats) and / or out_rgb8 (H*W*3 bytes: normalize() + to_vec() of the output rows by their own maximum);
 * stats: max_value, ms_render (device time of the traced and resolved rows: no tone map, no copies), ms_total,
 * kernel_launches, resident_prims, d2h_bytes.  Device memory: the output rows only (no s^2-sized scratch).  The call writes
 * the caller's float frame, so the library forgets its previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: a NULL lens, samples outside [1, 8], aperture < 0, focus <= 0, a lens value that is not finite;
 * an invalid view; precision other than RM_FP32; patch_row_stride > 1; max_depth < 1; an unknown scene; out_rgb and out_rgb8
 * both NULL.  RM_ERR_DIMENSIONS: as for rm_render_supersampled.  Lens and parameter errors are reported without a device.
 * Out of scope: random or per-pixel lens patterns and bokeh shapes; a lens for rm_render_adaptive, rm_render_dispersive,
 * rm_render_rows_* and rm_render_frame; an FP64 entry point.  A lens together with area lights, rough glass and motion:
 * rm_render_distributed. */
typedef struct RmLens {
    double aperture;   /* lens radius in scene units, >= 0 */
    double focus;      /* distance from the camera to the plane in focus, along the view axis, > 0 */
    int32_t samples;   /* s: s x s sample rays per pixel, in [1, 8] */
} RmLens;
int rm_render_lens(RmScene scene, const RmParams* params, const RmView* view, const RmLens* lens, float* out_rgb,
                   uint8_t* out_rgb8, RmStats* stats);

/* ---- extension mode: soft shadows -- spherical area lights ------------------------------------------------------------------ *
 * The reference's lights are points, so every shadow has a hard edge.  This call gives each of the scene's lights a radius
 * for one frame (the uploaded scene and its format do not change); a light of radius r > 0 casts a penumbra.
 * Definition (normative; rm::light_frame / rm::light_sample in rm_trace.cuh are this in f64, and the tests' restatement over
 * the oracle is the same).  Light l has position c, colour k, intensity I, radius r >= 0; s = samples.  The reference's
 * direct_lighting (renderer.rs:138-193) runs at every shading point p with unit normal n, at every recursion level; lights
 * are visited in scene order, as in the reference.
 *   - r = 0: the reference's point light: its own term, one shadow ray.
 *   - r > 0: the light is replaced at p by s^2 point lights q_ab, visited a = 0..s-1 (outer), b = 0..s-1 (inner).  Each
 *     contributes exactly the reference's per-light term with position q_ab and colour k * (1 / (s*s)): light_dir =
 *     normalized(q - p), side, the +-1e-3 shadow origin, the any-hit query with no maximum distance (an occluder beyond q
 *     still shadows, as in the reference), then diffuse and specular added to the running sum in that order.
 *   - Sample points, in f64 without fused multiply-add (Duff et al. 2017, "Building an orthonormal basis, revisited":
 *     branch-free and defined for every unit m):
 *       m = normalized(c - p)  (the reference's light_dir towards the centre);
 *       sigma = copysign(1, m.z);  alpha = -1 / (sigma + m.z);  beta = (m.x*m.y) * alpha;
 *       t1 = (1 + ((sigma*m.x)*m.x) * alpha, sigma*beta, -sigma*m.x);  t2 = (beta, sigma + (m.y*m.y) * alpha, -m.y);
 *       (lx, ly) = rm::lens_offset(s, a, b)  (RmLens's unit-disc points, as they are);
 *       q = c + r * ((lx*t1) + (ly*t2)), component by component in that order.
 *     The points lie on the disc of radius r through c that faces p: the silhouette of a spherical light.
 * Consequences:
 *   - At s = 1 the only point is (0, 0): q = c and the colour is k, both exactly -- the reference's frame.  A call whose
 *     radii are all 0 is the reference's frame as well.  Both are routed to rm_render and give its frame, ids and 8-bit
 *     frame bit for bit.
 *   - Primary visibility does not depend on the lights: out_prim_id is rm_render's, and lights stay invisible.
 * FP32 production path (area_light_kernel): primary hits as rm_render's kernel finds them (the same device functions);
 * m, t1, t2, q and the colour scale in FP32 from the FP32 shading point, every shadow ray through the FP32 any-hit query
 * (brute force, or the hierarchy with accel != 0 and at most 8 lights; accel = 2 renders as accel = 1); frames meet the FP32
 * parity criteria against the f64 definition.  cull_backfacing applies.  The cost grows with s^2 times the area lights.
 * Rows, outputs and stats as rm_render_lens: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched; out_rgb
 * (H*W*3 floats) and / or out_rgb8 (H*W*3 bytes: normalize() + to_vec() of the output rows by their own maximum); out_prim_id
 * (H*W, optional): rm_render's primary ids; stats: max_value, ms_render (device time of K0 and the traced rows: no tone map,
 * no copies), ms_total, kernel_launches, resident_prims, d2h_bytes; no event counters.  Device memory: the output rows (and
 * 4 bytes per light).  The call writes the caller's float frame, so the library forgets its previous deliveries into that
 * memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: a NULL lights; a NULL radius with n_lights > 0; a radius that is negative or not finite; samples
 * outside [1, 8]; precision other than RM_FP32; patch_row_stride > 1; max_depth < 1; out_rgb and out_rgb8 both NULL (all
 * reported without a device); n_lights different from the scene's light count; an unknown scene.  RM_ERR_DIMENSIONS: as
 * for rm_render.
 * Out of scope: area lights with a view, a lens, supersampling, rm_render_adaptive, rm_render_dispersive, rm_render_rows_*
 * or rm_render_frame; an FP64 entry point; random or per-pixel sampling patterns; shapes other than the facing disc; a
 * radius stored in the scene.  Area lights with a view, a lens, rough glass or motion, sampled one point per sample ray:
 * rm_render_distributed. */
typedef struct RmAreaLights {
    int32_t       n_lights;  /* must equal the scene's light count */
    const double* radius;    /* n_lights radii in the scene's light order: finite, >= 0 (0 = the reference's point light) */
    int32_t       samples;   /* s in [1, 8] */
} RmAreaLights;
int rm_render_area_lights(RmScene scene, const RmParams* params, const RmAreaLights* lights, float* out_rgb, int32_t* out_prim_id,
                          uint8_t* out_rgb8, RmStats* stats);

/* ---- extension mode: rough glass -- blurred refraction and reflection ------------------------------------------------------ *
 * The reference's glass refracts and reflects along ideal directions (optics.rs:8-89).  This call gives each primitive a
 * roughness for one frame (the uploaded scene and its format do not change): every ray a rough glass-like hit spawns is
 * spread over a cone, sampled s x s per pixel -- frosted glass.  reflect_ray spawns a ray only at total internal reflection,
 * so on glass the visible effect is mostly in the refracted ray; the roughness applies to both.
 * Definition (normative; rm::rough_dir / rm::rough_reflect_origin / rm::rough_refract_origin / rm::rough_offset in
 * rm_trace.cuh are this, and the tests' restatement over the oracle is the same).  All in f64 without fused multiply-add;
 * s = samples.
 *   1. Sample (i, j) of output pixel (x, y), i, j in [0, s), is rm_render_lens's sample ray: rm::lens_ray with the view's
 *      basis (the identity without a view) and the lens (aperture 0 without one).
 *   2. The sample's value is the reference's cast_ray from that ray (renderer.rs:254-309, levels 1..max_depth) with one
 *      change.  At a hit of recursion level L (1 = the sample ray's own hit) on a glass-like primitive k with
 *      g = roughness[k] > 0, let (lx, ly) = rm::lens_offset(s, (j + L) mod s, i) -- stratum ((i + j + L) mod s, i), a bijection
 *      over the s^2 samples at every level, different from the lens's strata and shifted per level.  If (lx, ly) != (0, 0),
 *      each ray the reference spawns there (reflect_ray's and refract_ray's, whichever exist) is changed:
 *        (t1, t2) = the basis of rd by RmAreaLights's formula (Duff et al. 2017) with m = rd;
 *        rd' = normalized(rd + g * ((lx*t1) + (ly*t2))), component by component in that order (geometry.rs's scale(1/norm));
 *        the origin by the producing function's own rule applied to rd': a reflected ray leaves from point - hit_normal*1e-4
 *        if dot(rd', hit_normal) < 0, else from point + hit_normal*1e-4; a refracted ray, with `normal` the hit normal turned
 *        against the incident ray, from point + normal*1e-4 if dot(rd', normal) > 0, else from point - normal*1e-4.
 *      Whether a ray exists (total internal reflection) and the weights k and 1 - k are decided before the change, exactly as
 *      the reference decides them.
 *   3. The pixel is the FP32 mean of its s^2 sample values in rm_render_supersampled's order (sub-rows i outer, j inner).
 * Consequences:
 *   - The offset is orthogonal to rd and at most 1 long, so rd' is always defined and lies within atan(g) of rd: g is the
 *     tangent of the blur cone's half-angle.
 *   - g = 0, or an offset of (0, 0), leaves the ray bit for bit as the reference spawns it; at s = 1 the only offset is (0, 0).
 *   - s = 1, all roughness 0, and roughness on no glass-like primitive (decided on the host from the scene's materials) give
 *     rm_render_lens's frame bit for bit and are routed there (which routes aperture 0 without a view to
 *     rm_render_supersampled).
 *   - Primary visibility does not depend on roughness: only rays spawned at glass-like hits turn.
 *   - The pattern is fixed per pixel, not random: the frame is deterministic.
 * FP32 production path (rough_glass_kernel): lens_kernel's schedule; each sample ray from rm::lens_ray in f64, traced with the
 * general FP32 closest-hit query (brute force, or the hierarchy with accel != 0; accel = 2 renders as accel = 1), the
 * recursion with a roughness per primitive id in FP32 (a positive value too small for FP32 is kept at 1e-30).  The turn is
 * computed in f64 from the f64 ray where the scene takes f64 ray geometry, in FP32 otherwise; frames meet the FP32 parity
 * criteria against the f64 definition.  cull_backfacing applies.
 * Rows, outputs and stats as rm_render_lens: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched; out_rgb
 * (H*W*3 floats) and / or out_rgb8 (H*W*3 bytes: normalize() + to_vec() of the output rows by their own maximum); stats:
 * max_value, ms_render, ms_total, kernel_launches, resident_prims, d2h_bytes.  Device memory: the output rows and 4 bytes per
 * primitive.  The call writes the caller's float frame, so the library forgets its previous deliveries into that memory
 * (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: a NULL rough; n_prims < 0, or a NULL roughness with n_prims > 0; a roughness that is negative or
 * not finite; samples outside [1, 8]; an invalid view or lens by rm_render_lens's rules; lens->samples != rough->samples;
 * precision other than RM_FP32; patch_row_stride > 1; max_depth < 1; out_rgb and out_rgb8 both NULL (all reported without
 * a device); n_prims different from rm_scene_num_prims(scene); an unknown scene.  RM_ERR_DIMENSIONS: as for
 * rm_render_supersampled.
 * Out of scope: rm_render_adaptive, rm_render_dispersive, rm_render_rows_* or rm_render_frame; an FP64 entry point; random
 * or per-pixel patterns and lobes other than the uniform-disc cone; roughness stored in the uploaded scene; per-channel
 * roughness.  Roughness with area lights or motion: rm_render_distributed. */
typedef struct RmRoughGlass {
    int32_t       n_prims;    /* must equal rm_scene_num_prims(scene) */
    const double* roughness;  /* n_prims values in primitive-id order (shapes in scene order, an Obj once per triangle):
                                 finite, >= 0; 0 = the reference's ideal refraction / reflection.  Read only for glass-like
                                 primitives: opaque hits spawn no ray (renderer.rs:277) */
    int32_t       samples;    /* s in [1, 8] */
} RmRoughGlass;
int rm_render_rough_glass(RmScene scene, const RmParams* params, const RmView* view /* NULL = the reference's camera */,
                          const RmLens* lens /* NULL = pinhole */, const RmRoughGlass* rough, float* out_rgb,
                          uint8_t* out_rgb8, RmStats* stats);

/* ---- extension mode: motion blur -- primitives that move over the shutter interval ------------------------------------------ *
 * The reference renders one instant.  This call gives each primitive a displacement for one frame (the uploaded scene and its
 * format do not change): over the shutter it moves by that much, and the s x s samples of a pixel see it at s^2 different
 * times -- moving objects smear along their path.  Translation only; lights and the camera do not move.
 * Definition (normative; rm::motion_time in rm_trace.cuh is this, and the tests' restatement over the oracle is the same).  All
 * in f64 without fused multiply-add; s = samples.
 *   1. Motion.  Primitive k (primitive-id order: shapes in scene order, an Obj once per triangle) has the displacement v_k
 *      (3 doubles): how far it moves over the whole shutter.  The uploaded scene is its pose at shutter time tau = 0.
 *   2. Time of a sample.  Sample (i, j), i, j in [0, s), of output pixel (x, y) has the time stratum
 *      m = s*((2i + j) mod s) + ((i + j) mod s) -- a bijection onto [0, s^2) for every s, since (a - b) mod s = i -- and the time
 *      tau = (m + 0.5) / s^2 - 0.5, in (-1/2, 1/2) and symmetric about 0.  Every pixel uses the same pattern.
 *   3. Scene at tau.  Primitive k is translated by tau*v_k, component by component: a sphere's centre becomes c + tau*v; a
 *      triangle's or polygon's vertices (and its plane point) become each vertex + tau*v, its normal unchanged.  Translation
 *      leaves normals alone, so the reference's world-z inside test and the hittable / back-facing / degenerate classes of a
 *      planar primitive do not change.
 *   4. The sample's value is the reference's cast_ray (renderer.rs:254-309, levels 1..max_depth) from rm_render_lens's sample
 *      ray (rm::lens_ray with the view's basis -- the identity without a view -- and the lens -- aperture 0 without one), in the
 *      scene at tau: the whole recursion and every shadow ray of the sample see the same tau.
 *   5. The pixel is the FP32 mean of its s^2 sample values in rm_render_supersampled's order (sub-rows i outer, j inner).
 * Consequences:
 *   - At s = 1, tau = 0; with every displacement zero nothing moves.  Both give rm_render_lens's frame bit for bit and are
 *     routed there (which routes aperture 0 without a view to rm_render_supersampled).
 *   - A pixel none of whose samples meets a swept primitive -- directly, through the recursion or through a shadow ray -- is
 *     rm_render_lens's pixel.
 *   - The pattern is fixed, not random: the frame is deterministic.
 * FP32 production path (motion_kernel): lens_kernel's schedule; each sample ray from rm::lens_ray in f64, each query at the
 * sample's tau: primitive k is tested against the ray with its origin shifted to o - tau*v_k (v_k rounded to FP32) -- the same
 * ray parameter t, and the unchanged per-primitive routines.  Brute force, or with accel != 0 a hierarchy over swept boxes
 * (each primitive's box at tau = -1/2 united with its box at tau = +1/2), built on the host once per scene and displacements
 * and kept (accel = 2 renders as accel = 1).  Frames meet the FP32 parity criteria against the f64 definition.
 * cull_backfacing applies.
 * Rows, outputs and stats as rm_render_lens: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched; out_rgb
 * (H*W*3 floats) and / or out_rgb8 (H*W*3 bytes: normalize() + to_vec() of the output rows by their own maximum); stats:
 * max_value, ms_render, ms_total, kernel_launches, resident_prims, d2h_bytes.  Device memory: the output rows, 16 bytes per
 * primitive and, with accel != 0, the swept hierarchy.  The call writes the caller's float frame, so the library forgets its
 * previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: a NULL motion; n_prims < 0, or a NULL displacement with n_prims > 0; a displacement that is not
 * finite; samples outside [1, 8]; an invalid view or lens by rm_render_lens's rules; lens->samples != motion->samples;
 * precision other than RM_FP32; patch_row_stride > 1; max_depth < 1; out_rgb and out_rgb8 both NULL (all reported without a
 * device); n_prims different from rm_scene_num_prims(scene); an unknown scene.  RM_ERR_DIMENSIONS: as for
 * rm_render_supersampled.
 * Out of scope: rm_render_adaptive, rm_render_dispersive, rm_render_rows_* or rm_render_frame; moving lights or a moving
 * camera; rotation, scaling or curved paths; motion stored in the uploaded scene; an FP64 entry point; random or per-pixel
 * time patterns.  Motion with rough glass or area lights: rm_render_distributed. */
typedef struct RmMotion {
    int32_t       n_prims;       /* must equal rm_scene_num_prims(scene) */
    const double* displacement;  /* 3 * n_prims values, x y z per primitive id (shapes in scene order, an Obj once per
                                    triangle): finite; how far the primitive moves over the shutter */
    int32_t       samples;       /* s in [1, 8] */
} RmMotion;
int rm_render_motion(RmScene scene, const RmParams* params, const RmView* view /* NULL = the reference's camera */,
                     const RmLens* lens /* NULL = pinhole */, const RmMotion* motion, float* out_rgb, uint8_t* out_rgb8,
                     RmStats* stats);

/* ---- extension mode: distributed ray tracing -- depth of field, soft shadows, rough glass and motion blur at once ---------- *
 * Cook, Porter and Carpenter (1984): every sample ray samples every dimension at once -- the lens point, the time, a point
 * of each area light and the direction of every ray rough glass scatters -- and the pixel is the mean over its samples.  This
 * call takes the structs of rm_render_lens, rm_render_area_lights, rm_render_rough_glass and rm_render_motion together; none
 * changes, and the ABI version stays 5.
 * Definition (normative; rm::area_offset in rm_trace.cuh holds rule 4's stratum, and the tests' restatement over the oracle is
 * the same).  All in f64 without fused multiply-add; s = samples, and every struct given has samples == s.
 *   1. Sample (i, j), i, j in [0, s), of output pixel (x, y) is rm_render_lens's sample ray: rm::lens_ray with the view's basis
 *      (the identity without a view) and the lens (aperture 0 without one).
 *   2. Time.  tau = rm::motion_time(s, i, j), and the sample sees the scene at tau as RmMotion defines it (without motion tau
 *      plays no role).  The whole recursion and every shadow ray of the sample see the same tau; lights and the camera do not
 *      move.
 *   3. Rough glass.  At a hit of level L, the rays a glass-like hit spawns are turned as RmRoughGlass defines it, with
 *      rm::rough_offset(s, i, j, L) and the same side rules for the origin; hit points and normals are the scene's at tau.
 *   4. Area lights, one point per sample.  At a shading point p of level L, a light of radius 0 is the reference's point
 *      light.  A light of centre c, colour k and radius r > 0 is ONE point light of colour k (not k / s^2) at
 *      q = rm::light_sample(c, r, t1, t2, lx, ly), with (t1, t2) = rm::light_frame(normalized(c - p)) and (lx, ly) the
 *      elliptical grid-to-disc map (rm::lens_offset's) of the stratum (a, b) = ((i + 2j + L) mod s, (i + 3j) mod s):
 *      rm::area_offset(s, i, j, L).  Its shadow ray is traced in the scene at tau; otherwise the term is the reference's
 *      per-light term, with the +-1e-3 origin and no maximum distance.  The stratum map has determinant 1 over Z_s, a bijection
 *      over the s^2 samples for every s and L; for s >= 4 neither coordinate is a shifted copy of a coordinate of the
 *      sub-pixel, lens, rough or time strata (at s = 2 and 3 some sharing cannot be avoided).
 *      This is NOT rm_render_area_lights' frame: there each pixel traces one primary ray and every area light is s^2 point
 *      lights of colour k / s^2 at each shading point.  Here the pixel's s^2 samples do the averaging, at s^2 shadow rays per
 *      area light and pixel instead of s^4.
 *   5. The pixel is the FP32 mean of its s^2 sample values in rm::resolve_box's order (sub-rows i outer, j inner).
 * Routing -- each routed case is that call, and gives its frame bit for bit.  An area light is active when its radius is
 * > 0; rough glass when some glass-like primitive has roughness > 0 (decided on the host, as rm_render_rough_glass does);
 * motion when some displacement is != 0.
 *   - s = 1, or no active effect: rm_render_lens (with the pinhole when no lens is given);
 *   - rough glass alone: rm_render_rough_glass;  motion alone: rm_render_motion;
 *   - an active area light, or rough glass together with motion: distributed_kernel.
 * FP32 production path (distributed_kernel): motion_kernel's schedule; queries at the sample's tau as rm_render_motion makes
 * them (over the swept hierarchy with accel != 0) when motion is active, and over the scene's own otherwise (brute force for
 * scenes of more than 8 lights); rough_glass_kernel's turn; the light point of rule 4 in FP32 from the FP32 shading point.
 * Frames meet the FP32 parity criteria against the f64 definition.  cull_backfacing applies.
 * Rows, outputs and stats as rm_render_lens: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched; out_rgb
 * and / or out_rgb8; stats: max_value, ms_render, ms_total, kernel_launches, resident_prims, d2h_bytes.  The call writes the
 * caller's float frame, so the library forgets its previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: samples outside [1, 8]; a given struct whose samples differs from s; a struct that is invalid by
 * its own call's rules (a radius, a roughness, a displacement, the view, the lens); precision other than RM_FP32;
 * patch_row_stride > 1; max_depth < 1; out_rgb and out_rgb8 both NULL (all reported without a device); n_lights different
 * from the scene's light count, n_prims different from rm_scene_num_prims(scene); an unknown scene.  RM_ERR_DIMENSIONS: as
 * for rm_render_supersampled.
 * Out of scope: random or per-pixel patterns; an FP64 entry point; combining with rm_render_adaptive, rm_render_dispersive,
 * rm_render_rows_* or rm_render_frame; moving lights.  Diffuse interreflection with these effects: rm_render_path. */
int rm_render_distributed(RmScene scene, const RmParams* params, int samples,
                          const RmView* view /* NULL = the reference's camera */, const RmLens* lens /* NULL = pinhole */,
                          const RmAreaLights* lights /* NULL = point lights */, const RmRoughGlass* rough /* NULL = ideal optics */,
                          const RmMotion* motion /* NULL = nothing moves */, float* out_rgb, uint8_t* out_rgb8, RmStats* stats);

/* ---- extension mode: diffuse interreflection -- light that bounces off opaque surfaces ------------------------------------- *
 * The reference's opaque hits add background + direct lighting and spawn no ray (renderer.rs:277), so a surface receives
 * light only from the lights it sees.  This call lets every opaque hit spawn one cosine-weighted diffuse ray per sample
 * (Kajiya 1986): colour bleeds from one surface onto its neighbours, and corners that see less of the scene darken.  No
 * scene data is added: the bounce's weight is the material's own diffusion * diffuse_color, the factor direct_lighting
 * applies (renderer.rs:181-183,192).  The ABI version stays 5.
 * Definition (normative; rm::diffuse_offset / rm::diffuse_point / rm::diffuse_stratum / rm::diffuse_normal / rm::diffuse_dir /
 * rm::diffuse_origin in rm_trace.cuh are this, and the tests' restatement over the oracle is the same).  All in f64 without
 * fused multiply-add; s = samples.
 *   1. Sample (i, j), i, j in [0, s), of output pixel (x, y) is rm_render_lens's sample ray: rm::lens_ray with the view's basis
 *      (the identity without a view) and the lens (aperture 0 without one).
 *   2. The sample's value is the reference's cast_ray from that ray (renderer.rs:254-309, levels 1..max_depth, the reference's
 *      order of additions) with one change.  At a hit of level L < max_depth on a primitive that is not glass-like, whose
 *      diffusion is > 0 and some of whose diffuse_color components are > 0, the sample spawns one diffuse ray:
 *        stratum: (a, b) = ((2i + 3j + L) mod s, (3i + 5j) mod s) -- determinant 2*5 - 3*3 = 1 over Z_s, a bijection over the
 *          s^2 samples for every s and L; for s >= 4 neither coordinate is a shifted copy of a coordinate of the sub-pixel,
 *          lens, rough, area or time strata (at s = 2 and 3 some sharing cannot be avoided);
 *        disc point: the Shirley-Chiu concentric map of the stratum centre, p = (2a + 1)/s - 1, q = (2b + 1)/s - 1: (0, 0) if
 *          p = q = 0; else if |p| > |q|, r = p and phi = (pi/4)(q/p); otherwise r = q and phi = pi/2 - (pi/4)(p/q);
 *          (lx, ly) = (r cos phi, r sin phi).  The map is equal-area, so Malley's lift below is cosine-weighted (the elliptical
 *          map of rm::lens_offset is not, and would weight the hemisphere wrongly);
 *        direction: n_f = the hit normal turned against the incident ray d (n if dot(n, d) < 0, else -n); (t1, t2) =
 *          rm::light_frame(n_f); z = sqrt(1 - ((lx lx) + (ly ly))), > 0 since r <= 1 - 1/s;
 *          rd = normalized(((lx t1) + (ly t2)) + z n_f), component by component in that order;
 *        origin: point + n_f 1e-4, reflect_ray's offset (optics.rs:41-45);
 *        addition: c = background + direct as the reference has it, then c += scaled(v * diffuse_color, diffusion), with v the
 *          value of the diffuse ray at level L + 1 (a miss there is the background, as for every level > 1).
 *      Glass-like hits keep the reference's optics and spawn no diffuse ray, so a level pushes at most one frame and max_depth
 *      caps the whole path, bounces included.
 *   3. The pixel is the FP32 mean of its s^2 sample values in rm::resolve_box's order (sub-rows i outer, j inner).
 * Consequences:
 *   - Primary visibility is rm_render_lens's.  At s = 1 every hit bounces once, along n_f.
 *   - The pattern is fixed per pixel, not random: the frame is deterministic, and under-sampled indirect light shows as
 *     structure, not noise.
 *   - max_depth = 1, and scenes in which no primitive meets the bounce condition (decided on the host from the scene's
 *     materials), give rm_render_lens's frame bit for bit and are routed there.  s = 1 is not routed.
 * FP32 production path (indirect_kernel): lens_kernel's schedule; each sample ray from rm::lens_ray in f64, traced with the
 * general FP32 closest-hit query (brute force, or the hierarchy with accel != 0 for scenes of at most 8 lights; accel = 2
 * renders as accel = 1).  The disc points are computed on the host (cos and sin) and read from a table; the bounce is computed
 * in f64 from the refined f64 point and normal where the scene takes f64 ray geometry, in FP32 otherwise.  Frames meet the FP32
 * parity criteria against the f64 definition.  cull_backfacing applies.
 * Rows, outputs and stats as rm_render_lens: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched; out_rgb
 * and / or out_rgb8; stats: max_value, ms_render, ms_total, kernel_launches, resident_prims, d2h_bytes.  The call writes the
 * caller's float frame, so the library forgets its previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: samples outside [1, 8]; an invalid view or lens by rm_render_lens's rules; lens->samples !=
 * samples; precision other than RM_FP32; patch_row_stride > 1; max_depth < 1; out_rgb and out_rgb8 both NULL (all reported
 * without a device); an unknown scene.  RM_ERR_DIMENSIONS: as for rm_render_supersampled.
 * Out of scope: combining with rm_render_distributed (area lights, rough glass, motion); bounces from glass-like hits;
 * emissive materials; random or per-pixel patterns and progressive accumulation; an FP64 entry point; rm_render_rows_*,
 * rm_render_frame, rm_render_adaptive or rm_render_dispersive.  The bounce with area lights, rough glass and motion:
 * rm_render_path. */
int rm_render_indirect(RmScene scene, const RmParams* params, const RmView* view /* NULL = the reference's camera */,
                       const RmLens* lens /* NULL = pinhole */, int samples, float* out_rgb, uint8_t* out_rgb8, RmStats* stats);

/* ---- extension mode: path-traced frames -- diffuse interreflection with depth of field, soft shadows, rough glass and
 * motion blur at once ------------------------------------------------------------------------------------------------------ *
 * rm_render_indirect's diffuse bounce inside rm_render_distributed's frame: every sample ray samples the lens point, the time,
 * a point of each area light, the turn of every ray rough glass spawns and the direction of every diffuse ray, and the pixel
 * is the mean over its samples (Cook 1984 with Kajiya 1986's bounce).  The signature is rm_render_distributed's; no struct is
 * added or changed, and the ABI version stays 5.
 * Definition (normative; every rule is already stated above for rm_render_lens, rm_render_motion, rm_render_rough_glass,
 * rm_render_distributed and rm_render_indirect, and the tests' restatement over the oracle is the same).  All in f64 without
 * fused multiply-add; s = samples, and every struct given has samples == s.
 *   1. Sample ray.  Sample (i, j), i, j in [0, s), of output pixel (x, y) is rm_render_lens's sample ray: rm::lens_ray with the
 *      view's basis (the identity without a view) and the lens (aperture 0 without one).
 *   2. Time.  tau = rm::motion_time(s, i, j), and the sample sees the scene at tau as RmMotion defines it.  Every query of the
 *      sample's path sees the same tau: primary, glass, diffuse and shadow rays alike.  Lights and the camera do not move.
 *   3. Rough glass.  The rays a rough glass-like hit of level L spawns are turned with rm::rough_offset(s, i, j, L), as in
 *      rm_render_distributed rule 3.
 *   4. Area lights.  At every shading point of level L, a light of radius r > 0 is one point light of its full colour at the
 *      point of stratum rm::area_offset(s, i, j, L), as in rm_render_distributed rule 4.  The hit of a diffuse ray spawned at
 *      level L is a shading point of level L + 1, so it samples its lights at rm::area_offset(s, i, j, L + 1).
 *   5. Diffuse bounce.  rm_render_indirect rule 2, unchanged: at a hit of level L < max_depth on a primitive that is not
 *      glass-like, whose diffusion is > 0 and some of whose diffuse_color components are > 0, one diffuse ray of stratum
 *      rm::diffuse_stratum(s, i, j, L), through the concentric disc map and rm::diffuse_dir, from rm::diffuse_origin; the point
 *      and normal are the scene's at tau.  The additions are, in this order: c = background + direct(L); then, if glass-like,
 *      the reference's reflect / refract terms; otherwise c += scaled(v * diffuse_color, diffusion).
 *   6. The pixel is the FP32 mean of its s^2 sample values in rm::resolve_box's order (sub-rows i outer, j inner).
 * Glass-like hits spawn no diffuse ray, so a level pushes at most one frame and max_depth caps the whole path.
 * Routing -- each routed case is that call, and gives its frame bit for bit.  "Active" is as rm_render_distributed has it: a
 * radius > 0, roughness > 0 on a glass-like primitive, a displacement != 0.
 *   - max_depth = 1, or no primitive meets the bounce condition (decided on the host from the scene's materials):
 *     rm_render_distributed with the same arguments (which routes further by itself);
 *   - otherwise s = 1 (area_offset, rough_offset and motion_time are then the identity), or no active effect:
 *     rm_render_indirect(scene, params, view, lens, s, ...);
 *   - otherwise path_kernel.
 * FP32 production path (path_kernel): distributed_kernel's schedule, with rm_render_distributed's queries (at the sample's tau
 * over the swept hierarchy with accel != 0 when motion is active, over the scene's own otherwise; brute force for scenes of
 * more than 8 lights), its light points and its rough turn, and rm_render_indirect's bounce: read from the host's disc-point
 * table, computed in f64 from the refined f64 point (at tau with motion) and normal where the scene takes f64 ray geometry, in
 * FP32 otherwise.  Frames meet the FP32 parity criteria against the f64 definition.  cull_backfacing applies.
 * Rows, outputs and stats as rm_render_distributed: patch rows [b, e) with patch_row_stride <= 1, rows outside untouched;
 * out_rgb and / or out_rgb8; stats: max_value, ms_render, ms_total, kernel_launches, resident_prims, d2h_bytes.  The call
 * writes the caller's float frame, so the library forgets its previous deliveries into that memory (RM_ROWS_RETAINED).
 * RM_ERR_INVALID_ARGUMENT: as for rm_render_distributed, with the same messages for the structs (reported without a device,
 * except the light and primitive counts); an unknown scene.  RM_ERR_DIMENSIONS: as for rm_render_supersampled.
 * Out of scope: bounces from glass-like hits; emissive materials and sampling emitters by their geometry; random, per-pixel or
 * progressive sample patterns and s > 8; an FP64 entry point; rm_render_rows_*, rm_render_frame, rm_render_adaptive or
 * rm_render_dispersive; moving lights. */
int rm_render_path(RmScene scene, const RmParams* params, int samples, const RmView* view /* NULL = the reference's camera */,
                   const RmLens* lens /* NULL = pinhole */, const RmAreaLights* lights /* NULL = point lights */,
                   const RmRoughGlass* rough /* NULL = ideal optics */, const RmMotion* motion /* NULL = nothing moves */,
                   float* out_rgb, uint8_t* out_rgb8, RmStats* stats);

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
