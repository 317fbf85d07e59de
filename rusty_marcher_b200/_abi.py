"""ctypes binding of the C ABI (include/rm_b200.h, include/rm_b200_host.h).

The shared library is built in-tree by rusty_marcher_b200.build (nvcc, sm_100a).  There is no
CPU fallback: if the library is missing or no sm_100 GPU is present, loading/initialising raises.
"""
import ctypes as C
import os

from . import build as _build

d3 = C.c_double * 3


class RmReflectance(C.Structure):
    _fields_ = [("diffusion", C.c_double), ("diffuse_color", d3), ("specular", C.c_double),
                ("specular_exponent", C.c_double), ("is_glass_like", C.c_int32), ("reflection", C.c_double),
                ("refractive_index", C.c_double)]


class RmSphere(C.Structure):
    _fields_ = [("center", d3), ("radius_square", C.c_double), ("reflectance", RmReflectance)]


class RmPolygon(C.Structure):
    _fields_ = [("first_vertex", C.c_int32), ("n_vertices", C.c_int32), ("plane_normal", d3), ("plane_point", d3),
                ("reflectance", RmReflectance)]


class RmTriangle(C.Structure):
    _fields_ = [("vertices", C.c_double * 9), ("normal", d3), ("center", d3)]


class RmObj(C.Structure):
    _fields_ = [("first_triangle", C.c_int32), ("n_triangles", C.c_int32)]


class RmLight(C.Structure):
    _fields_ = [("position", d3), ("color", d3), ("intensity", C.c_double)]


class RmShapeRef(C.Structure):
    _fields_ = [("kind", C.c_int32), ("index", C.c_int32)]


class RmFlatScene(C.Structure):
    _fields_ = [("n_shapes", C.c_int32), ("shapes", C.POINTER(RmShapeRef)),
                ("n_spheres", C.c_int32), ("spheres", C.POINTER(RmSphere)),
                ("n_polygons", C.c_int32), ("polygons", C.POINTER(RmPolygon)),
                ("n_polygon_vertices", C.c_int32), ("polygon_vertices", C.POINTER(C.c_double)),
                ("n_objs", C.c_int32), ("objs", C.POINTER(RmObj)),
                ("n_triangles", C.c_int32), ("triangles", C.POINTER(RmTriangle)),
                ("triangle_reflectances", C.POINTER(RmReflectance)),
                ("n_lights", C.c_int32), ("lights", C.POINTER(RmLight))]


class RmParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("fov", C.c_double), ("camera", d3),
                ("max_depth", C.c_int32), ("background", C.c_double), ("patch_size", C.c_int32),
                ("precision", C.c_int32), ("patch_row_begin", C.c_int32), ("patch_row_end", C.c_int32),
                ("cull_backfacing", C.c_int32), ("patch_row_stride", C.c_int32), ("accel", C.c_int32)]


COUNTER_FIELDS = ["pixels", "closest_segments", "anyhit_segments", "sphere_tests", "sphere_disc", "sphere_hits",
                  "plane_tests", "plane_dist", "plane_point", "edge_tests", "cand_dist", "hits", "light_evals",
                  "lit_lights", "glass_hits", "reflections", "refractions"]


class RmStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in COUNTER_FIELDS] + [
        ("max_value", C.c_double), ("ms_render", C.c_double), ("ms_total", C.c_double),
        ("kernel_launches", C.c_int32), ("resident_prims", C.c_int32), ("d2h_bytes", C.c_uint64)]

    def counters(self):
        return {n: int(getattr(self, n)) for n in COUNTER_FIELDS}


RM_MAX_RANKS, RM_IPC_HANDLE_BYTES, RM_MAILBOX_BYTES = 16, 64, 512


class RmExchange(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("mailbox", C.c_void_p * RM_MAX_RANKS), ("frame8", C.c_void_p * 2)]


RM_FP32, RM_FP64 = 0, 1
RM_ROWS_RETAINED = 1
RM_OK = 0
STATUS_NAMES = {0: "RM_OK", -1: "RM_ERR_NO_DEVICE", -2: "RM_ERR_NOT_INITIALISED", -3: "RM_ERR_INVALID_ARGUMENT",
                -4: "RM_ERR_DIMENSIONS", -5: "RM_ERR_SCENE", -6: "RM_ERR_CUDA", -7: "RM_ERR_OUT_OF_MEMORY", -8: "RM_ERR_PEER"}

# every symbol include/rm_b200.h and include/rm_b200_host.h declare: name -> (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    "rm_abi_version": (C.c_int, []),
    "rm_init": (C.c_int, [C.c_int]),
    "rm_shutdown": (None, []),
    "rm_last_error": (C.c_char_p, []),
    "rm_device_info": (C.c_int, [C.c_char_p, C.c_int, _P(C.c_int), _P(C.c_int), _P(C.c_int), _P(C.c_int)]),
    "rm_params_default": (None, [_P(RmParams), C.c_int, C.c_int]),
    "rm_reflectance_default": (None, [_P(RmReflectance)]),
    "rm_scene_upload": (C.c_int, [_P(RmFlatScene), _P(C.c_int64)]),
    "rm_scene_free": (C.c_int, [C.c_int64]),
    "rm_scene_num_prims": (C.c_int, [C.c_int64]),
    "rm_render": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_render_f64": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_render_rows_f64": (C.c_int, [C.c_int64, _P(RmParams), _P(C.c_void_p), C.c_int, _P(RmStats)]),
    "rm_render_rows_f32": (C.c_int, [C.c_int64, _P(RmParams), _P(C.c_void_p), C.c_int, _P(RmStats)]),
    "rm_render_device": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rm_render_device_stats": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_render_device_rgb8": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rm_tonemap_device": (C.c_int, [_P(RmParams), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "rm_tonemap_device_busy": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "rm_set_profiling": (C.c_int, [C.c_int]),
    "rm_last_kernel_times": (C.c_int, [_P(C.c_double), _P(C.c_double)]),
    "rm_kernel_times": (C.c_int, [C.c_int, _P(C.c_double), _P(C.c_double), _P(C.c_double)]),
    "rm_render_dispersive": (C.c_int, [_P(C.c_int64), _P(RmParams), C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_render_supersampled": (C.c_int, [C.c_int64, _P(RmParams), C.c_int, C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_render_adaptive": (C.c_int, [C.c_int64, _P(RmParams), C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, _P(RmStats)]),
    "rm_scene_query_count": (C.c_int, [C.c_int64, _P(C.c_uint64), C.c_int]),
    "rm_scene_accel_status": (C.c_int, [C.c_int64, _P(C.c_int32)]),
    "rm_scene_walk_stats": (C.c_int, [C.c_int64, _P(C.c_uint64), C.c_int]),
    "rm_peer_alloc": (C.c_int, [C.c_size_t, _P(C.c_void_p), C.c_char_p]),
    "rm_peer_open": (C.c_int, [C.c_char_p, _P(C.c_void_p)]),
    "rm_peer_close": (C.c_int, [C.c_void_p]),
    "rm_peer_free": (C.c_int, [C.c_void_p]),
    "rm_render_frame": (C.c_int, [C.c_int64, _P(RmParams), C.c_void_p, C.c_void_p, C.c_void_p, _P(RmExchange), C.c_uint32, C.c_int, C.c_void_p]),
    "rm_peer_status": (C.c_int, [_P(RmExchange)]),
    "rm_graph_launch_count": (C.c_longlong, []),
    "rm_peer_stamps": (C.c_int, [_P(RmExchange), _P(C.c_uint64)]),
    "rm_content_hash": (C.c_uint64, [C.c_void_p, C.c_size_t, C.c_uint64]),
    "rm_host_alloc": (C.c_void_p, [C.c_size_t]),
    "rm_host_free": (None, [C.c_void_p]),
    "rm_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "rm_host_unregister": (C.c_int, [C.c_void_p]),
    "rm_measure_fp32_peak": (C.c_int, [_P(C.c_double), _P(C.c_double)]),
    # host builder
    "rm_builder_new": (C.c_void_p, []),
    "rm_builder_create_default": (C.c_void_p, []),
    "rm_builder_free": (None, [C.c_void_p]),
    "rm_builder_set_camera": (None, [C.c_void_p, _P(C.c_double)]),
    "rm_builder_offset_camera": (None, [C.c_void_p, _P(C.c_double)]),
    "rm_builder_get_camera": (None, [C.c_void_p, _P(C.c_double)]),
    "rm_builder_add_sphere": (C.c_int, [C.c_void_p, _P(C.c_double), C.c_double, _P(RmReflectance)]),
    "rm_builder_add_polygon": (C.c_int, [C.c_void_p, _P(C.c_double), C.c_int, _P(RmReflectance)]),
    "rm_builder_add_mesh": (C.c_int, [C.c_void_p, _P(C.c_double), C.c_int, _P(C.c_double)]),
    "rm_builder_add_triangles": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_char_p]),
    "rm_builder_add_obj_file": (C.c_int, [C.c_void_p, C.c_char_p, _P(C.c_double)]),
    "rm_builder_add_light": (None, [C.c_void_p, _P(C.c_double), _P(C.c_double), C.c_double]),
    "rm_builder_num_shapes": (C.c_int, [C.c_void_p]),
    "rm_builder_num_prims": (C.c_int, [C.c_void_p]),
    "rm_builder_shape_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "rm_builder_flatten": (_P(RmFlatScene), [C.c_void_p]),
    "rm_builder_upload": (C.c_int, [C.c_void_p, _P(C.c_int64)]),
    "rm_write_ppm": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


class RmError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("%s: %s" % (STATUS_NAMES.get(code, code), message))
        self.code = code


def lib_path():
    return _build.LIB


def load(build_if_missing=True):
    """Loads librm_b200.so (building it with nvcc if needed) and types every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("RM_B200_LIB") or _build.LIB           # RM_B200_LIB: another build of the same library (A/B runs)
    if build_if_missing and path == _build.LIB:
        _build.build()
    if not os.path.exists(path):
        raise RuntimeError("librm_b200.so is missing and could not be built; there is no CPU fallback")
    L = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)      # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise RmError(rc, load().rm_last_error().decode("utf-8", "replace"))
    return rc


_initialised_device = None


def init(device=0):
    """rm_init: binds this process to one GPU.  Raises RmError(RM_ERR_NO_DEVICE) without a B200."""
    global _initialised_device
    if _initialised_device == device:
        return
    check(load().rm_init(int(device)))
    _initialised_device = device


def shutdown():
    global _initialised_device
    if _lib is not None:
        _lib.rm_shutdown()
    _initialised_device = None
