//! ffi.rs -- the `extern "C"` boundary of the B200 render path: a field-for-field, symbol-for-symbol
//! transcription of `include/rm_b200.h` (ABI version 5).  `tests/test_integration_overlay.py` of the
//! rm_b200 repository parses this file and checks every struct's field order and every declared function
//! against the header.
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_void};

pub const RM_ABI_VERSION: c_int = 5;
pub const RM_OK: c_int = 0;
pub const RM_ERR_NO_DEVICE: c_int = -1;
pub const RM_ERR_NOT_INITIALISED: c_int = -2;
pub const RM_ERR_INVALID_ARGUMENT: c_int = -3;
pub const RM_ERR_DIMENSIONS: c_int = -4;
pub const RM_ERR_SCENE: c_int = -5;
pub const RM_ERR_CUDA: c_int = -6;
pub const RM_ERR_OUT_OF_MEMORY: c_int = -7;
pub const RM_ERR_PEER: c_int = -8;
pub const RM_FP32: i32 = 0;
pub const RM_FP64: i32 = 1;
pub const RM_SHAPE_SPHERE: i32 = 0;
pub const RM_SHAPE_POLYGON: i32 = 1;
pub const RM_SHAPE_OBJ: i32 = 2;
pub const RM_ROWS_RETAINED: c_int = 1;
pub const RM_MAX_RANKS: usize = 16;
pub const RM_IPC_HANDLE_BYTES: usize = 64;
pub const RM_MAILBOX_BYTES: usize = 512;

/// shapes.rs:21-32
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmReflectance {
    pub diffusion: f64,
    pub diffuse_color: [f64; 3],
    pub specular: f64,
    pub specular_exponent: f64,
    pub is_glass_like: i32,
    pub reflection: f64,
    pub refractive_index: f64,
}

/// sphere.rs:6-11
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmSphere {
    pub center: [f64; 3],
    pub radius_square: f64,
    pub reflectance: RmReflectance,
}

/// polygon.rs:6-12; the vertices live in RmFlatScene.polygon_vertices
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmPolygon {
    pub first_vertex: i32,
    pub n_vertices: i32,
    pub plane_normal: [f64; 3],
    pub plane_point: [f64; 3],
    pub reflectance: RmReflectance,
}

/// triangle.rs:6-10
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmTriangle {
    pub vertices: [f64; 9],
    pub normal: [f64; 3],
    pub center: [f64; 3],
}

/// obj.rs:14-20: a run of triangles + their reflectances
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmObj {
    pub first_triangle: i32,
    pub n_triangles: i32,
}

/// lights.rs:4-8
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmLight {
    pub position: [f64; 3],
    pub color: [f64; 3],
    pub intensity: f64,
}

/// one entry of Scene.shapes (scene.rs:11), in scene order
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmShapeRef {
    pub kind: i32,
    pub index: i32,
}

/// scene.rs:9-13, flattened; arrays are owned by the caller and copied by rm_scene_upload
#[repr(C)]
pub struct RmFlatScene {
    pub n_shapes: i32,
    pub shapes: *const RmShapeRef,
    pub n_spheres: i32,
    pub spheres: *const RmSphere,
    pub n_polygons: i32,
    pub polygons: *const RmPolygon,
    pub n_polygon_vertices: i32,
    pub polygon_vertices: *const f64,
    pub n_objs: i32,
    pub objs: *const RmObj,
    pub n_triangles: i32,
    pub triangles: *const RmTriangle,
    pub triangle_reflectances: *const RmReflectance,
    pub n_lights: i32,
    pub lights: *const RmLight,
}

#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmParams {
    pub width: i32,
    pub height: i32,
    pub fov: f64,
    pub camera: [f64; 3],
    pub max_depth: i32,
    pub background: f64,
    pub patch_size: i32,
    pub precision: i32,
    pub patch_row_begin: i32,
    pub patch_row_end: i32,
    pub cull_backfacing: i32,
    pub patch_row_stride: i32,
    pub accel: i32,
}

#[repr(C)]
#[derive(Copy, Clone, Debug, Default)]
pub struct RmStats {
    pub pixels: u64,
    pub closest_segments: u64,
    pub anyhit_segments: u64,
    pub sphere_tests: u64,
    pub sphere_disc: u64,
    pub sphere_hits: u64,
    pub plane_tests: u64,
    pub plane_dist: u64,
    pub plane_point: u64,
    pub edge_tests: u64,
    pub cand_dist: u64,
    pub hits: u64,
    pub light_evals: u64,
    pub lit_lights: u64,
    pub glass_hits: u64,
    pub reflections: u64,
    pub refractions: u64,
    pub max_value: f64,
    pub ms_render: f64,
    pub ms_total: f64,
    pub kernel_launches: i32,
    pub resident_prims: i32,
    pub d2h_bytes: u64,
}

pub type RmScene = i64;

/// camera orientation of rm_render_view: the basis is w = -forward, u = up x w, v = w x u (all normalised, f64)
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmView {
    pub forward: [f64; 3],
    pub up: [f64; 3],
}

/// thin-lens camera of rm_render_lens: lens radius (>= 0), distance of the plane in focus (> 0), s x s samples per pixel
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmLens {
    pub aperture: f64,
    pub focus: f64,
    pub samples: i32,
}

/// spherical area lights of rm_render_area_lights: one radius per scene light (0: the reference's point light), s x s samples
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmAreaLights {
    pub n_lights: i32,
    pub radius: *const f64,
    pub samples: i32,
}

/// rough glass of rm_render_rough_glass: one roughness per primitive id (0: the reference's ideal optics), s x s samples
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmRoughGlass {
    pub n_prims: i32,
    pub roughness: *const f64,
    pub samples: i32,
}

/// motion blur of rm_render_motion: one displacement (x, y, z) per primitive id over the shutter, s x s samples in time
#[repr(C)]
#[derive(Copy, Clone, Debug)]
pub struct RmMotion {
    pub n_prims: i32,
    pub displacement: *const f64,
    pub samples: i32,
}

/// one frame on the GPUs of one box (one process per GPU)
#[repr(C)]
pub struct RmExchange {
    pub rank: i32,
    pub world: i32,
    pub mailbox: [*mut c_void; RM_MAX_RANKS],
    pub frame8: [*mut u8; 2],
}

extern "C" {
    // ---- lifecycle
    pub fn rm_abi_version() -> c_int;
    pub fn rm_init(device: c_int) -> c_int;
    pub fn rm_shutdown();
    pub fn rm_last_error() -> *const c_char;
    pub fn rm_device_info(name: *mut c_char, name_len: c_int, sm_count: *mut c_int, cc_major: *mut c_int,
                          cc_minor: *mut c_int, clock_khz: *mut c_int) -> c_int;
    pub fn rm_params_default(p: *mut RmParams, width: c_int, height: c_int);
    pub fn rm_reflectance_default(r: *mut RmReflectance);
    // ---- scene
    pub fn rm_scene_upload(scene: *const RmFlatScene, out_handle: *mut RmScene) -> c_int;
    pub fn rm_scene_free(handle: RmScene) -> c_int;
    pub fn rm_scene_num_prims(handle: RmScene) -> c_int;
    // ---- the hot path, host buffers
    pub fn rm_render(scene: RmScene, params: *const RmParams, out_rgb: *mut f32, out_prim_id: *mut i32,
                     out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    pub fn rm_render_f64(scene: RmScene, params: *const RmParams, out_rgb: *mut f64, out_prim_id: *mut i32,
                         out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// rows[y] -> row y of FrameBuffer.buffer: width * 3 f64 (Vec<Vec3f> with #[repr(C)] Vec3f)
    pub fn rm_render_rows_f64(scene: RmScene, params: *const RmParams, rows: *const *mut f64, flags: c_int,
                              stats: *mut RmStats) -> c_int;
    pub fn rm_render_rows_f32(scene: RmScene, params: *const RmParams, rows: *const *mut f32, flags: c_int,
                              stats: *mut RmStats) -> c_int;
    pub fn rm_render_dispersive(scenes: *const RmScene, params: *const RmParams, out_rgb: *mut f32,
                                out_prim_id: *mut i32, stats: *mut RmStats) -> c_int;
    /// s x s samples per pixel (samples in [1, 8]): the s x frame box-filtered down to W x H
    pub fn rm_render_supersampled(scene: RmScene, params: *const RmParams, samples: c_int, out_rgb: *mut f32,
                                  out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// s x s samples only at the pixels the 3x3 id and contrast test refines, one sample elsewhere
    pub fn rm_render_adaptive(scene: RmScene, params: *const RmParams, samples: c_int, contrast: f64, out_rgb: *mut f32,
                              out_rgb8: *mut u8, out_mask: *mut u8, stats: *mut RmStats) -> c_int;
    /// u, v, w of a view (no GPU needed)
    pub fn rm_view_basis(view: *const RmView, out_basis: *mut f64) -> c_int;
    /// rm_render / rm_render_f64 / rm_render_device from the camera turned to `view`
    pub fn rm_render_view(scene: RmScene, params: *const RmParams, view: *const RmView, out_rgb: *mut f32,
                          out_prim_id: *mut i32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    pub fn rm_render_view_f64(scene: RmScene, params: *const RmParams, view: *const RmView, out_rgb: *mut f64,
                              out_prim_id: *mut i32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    pub fn rm_render_view_device(scene: RmScene, params: *const RmParams, view: *const RmView, d_rgb: *mut c_void,
                                 d_prim_id: *mut i32, d_max: *mut c_void, stream: *mut c_void) -> c_int;
    /// depth of field: s x s sample rays per pixel through a thin lens, from the camera turned to `view` (null: down -z)
    pub fn rm_render_lens(scene: RmScene, params: *const RmParams, view: *const RmView, lens: *const RmLens, out_rgb: *mut f32,
                          out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// soft shadows: every light of radius r > 0 as s x s points of the disc of radius r facing the shading point
    pub fn rm_render_area_lights(scene: RmScene, params: *const RmParams, lights: *const RmAreaLights, out_rgb: *mut f32,
                                 out_prim_id: *mut i32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// rough glass: the rays a glass-like hit spawns spread over a cone of half-angle atan(roughness), s x s samples per pixel
    pub fn rm_render_rough_glass(scene: RmScene, params: *const RmParams, view: *const RmView, lens: *const RmLens,
                                 rough: *const RmRoughGlass, out_rgb: *mut f32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// motion blur: every primitive translated by tau * displacement, the s x s samples of a pixel at s^2 times tau in (-1/2, 1/2)
    pub fn rm_render_motion(scene: RmScene, params: *const RmParams, view: *const RmView, lens: *const RmLens,
                            motion: *const RmMotion, out_rgb: *mut f32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// distributed ray tracing: lens, area lights (one point per sample ray), rough glass and motion together, s x s samples per
    /// pixel; every struct may be null, and every one given has samples == s
    pub fn rm_render_distributed(scene: RmScene, params: *const RmParams, samples: c_int, view: *const RmView, lens: *const RmLens,
                                 lights: *const RmAreaLights, rough: *const RmRoughGlass, motion: *const RmMotion,
                                 out_rgb: *mut f32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// diffuse interreflection: every qualifying opaque hit spawns one cosine-weighted diffuse ray per sample, s x s samples per
    /// pixel through the thin lens (null: pinhole) from the camera turned to `view` (null: down -z)
    pub fn rm_render_indirect(scene: RmScene, params: *const RmParams, view: *const RmView, lens: *const RmLens, samples: c_int,
                              out_rgb: *mut f32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    /// path-traced frames: rm_render_indirect's diffuse bounce with rm_render_distributed's lens, area lights, rough glass and
    /// motion (each null: left out), s x s samples per pixel
    pub fn rm_render_path(scene: RmScene, params: *const RmParams, samples: c_int, view: *const RmView, lens: *const RmLens,
                          lights: *const RmAreaLights, rough: *const RmRoughGlass, motion: *const RmMotion,
                          out_rgb: *mut f32, out_rgb8: *mut u8, stats: *mut RmStats) -> c_int;
    // ---- the hot path, device buffers
    pub fn rm_render_device(scene: RmScene, params: *const RmParams, d_rgb: *mut c_void, d_prim_id: *mut i32,
                            d_max: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn rm_render_device_rgb8(scene: RmScene, params: *const RmParams, d_rgb: *mut c_void, d_prim_id: *mut i32,
                                 d_max: *mut c_void, d_rgb8: *mut u8, stream: *mut c_void) -> c_int;
    pub fn rm_tonemap_device_busy(scene: RmScene, params: *const RmParams, d_rgb: *const c_void, d_max: *const c_void,
                                  normalise: c_int, d_rgb8: *mut u8, stream: *mut c_void) -> c_int;
    pub fn rm_render_device_stats(scene: RmScene, params: *const RmParams, d_rgb: *mut c_void, d_prim_id: *mut i32,
                                  d_max: *mut c_void, stream: *mut c_void, stats: *mut RmStats) -> c_int;
    pub fn rm_tonemap_device(params: *const RmParams, d_rgb: *const c_void, d_max: *const c_void, normalise: c_int,
                             d_rgb8: *mut u8, stream: *mut c_void) -> c_int;
    // ---- pinned host memory
    pub fn rm_content_hash(data: *const c_void, bytes: usize, seed: u64) -> u64;
    pub fn rm_host_alloc(bytes: usize) -> *mut c_void;
    pub fn rm_host_free(p: *mut c_void);
    pub fn rm_host_register(p: *mut c_void, bytes: usize) -> c_int;
    pub fn rm_host_unregister(p: *mut c_void) -> c_int;
    // ---- one frame on the GPUs of one box
    pub fn rm_peer_alloc(bytes: usize, d_ptr: *mut *mut c_void, handle: *mut u8) -> c_int;
    pub fn rm_peer_open(handle: *const u8, d_ptr: *mut *mut c_void) -> c_int;
    pub fn rm_peer_close(d_ptr: *mut c_void) -> c_int;
    pub fn rm_peer_free(d_ptr: *mut c_void) -> c_int;
    pub fn rm_render_frame(scene: RmScene, params: *const RmParams, d_rgb: *mut c_void, d_prim_id: *mut i32,
                           d_max: *mut c_void, exchange: *const RmExchange, seq: u32, normalise: c_int,
                           stream: *mut c_void) -> c_int;
    pub fn rm_peer_status(exchange: *const RmExchange) -> c_int;
    pub fn rm_graph_launch_count() -> i64;
    pub fn rm_peer_stamps(exchange: *const RmExchange, out_ns: *mut u64) -> c_int;
    // ---- measurement
    pub fn rm_set_profiling(on: c_int) -> c_int;
    pub fn rm_last_kernel_times(ms_prepare: *mut f64, ms_render: *mut f64) -> c_int;
    pub fn rm_kernel_times(back: c_int, ms_prepare: *mut f64, ms_render: *mut f64, ms_tonemap: *mut f64) -> c_int;
    pub fn rm_scene_query_count(scene: RmScene, out_queries: *mut u64, reset: c_int) -> c_int;
    pub fn rm_scene_walk_stats(scene: RmScene, out: *mut u64, reset: c_int) -> c_int;
    pub fn rm_scene_accel_status(scene: RmScene, out_words: *mut i32) -> c_int;
    pub fn rm_measure_fp32_peak(out_tflops: *mut f64, out_ms: *mut f64) -> c_int;
}

/// Turns a failed call into a panic (the reference's `render` has no error path: it panics, renderer.rs:107).
pub fn check(rc: c_int) {
    if rc != RM_OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(rm_last_error()) }.to_string_lossy().into_owned();
        panic!("rm_b200: {} ({})", msg, rc);
    }
}
