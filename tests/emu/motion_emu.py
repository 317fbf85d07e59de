"""ctypes binding of tests/emu/rm_motion_emu.cpp: rm_render_motion's per-ray kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from rusty_marcher_b200 import _abi

from . import emu
from .lens_emu import _basis, lens, params

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_motion_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_motion_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_motion_time.restype = C.c_double
        L.emu_motion_time.argtypes = [C.c_int, C.c_int, C.c_int]
        L.emu_render_motion.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.POINTER(_abi.RmLens), d,
                                        C.c_void_p, C.c_int]
        L.emu_swept_bvh.argtypes = [C.POINTER(_abi.RmFlatScene), d, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                    C.POINTER(C.c_int)]
        L.emu_set_glass_mode.argtypes = [C.c_int]
        _lib = L
    return _lib


def motion_time(s, i, j):
    return lib().emu_motion_time(s, i, j)


def _disp(disp):
    v = np.ascontiguousarray(disp, dtype=np.float64).reshape(-1, 3)
    return v, v.ctypes.data_as(C.POINTER(C.c_double))


def swept_bvh(scene, disp):
    """The swept hierarchy of the scene's FP32 pack under disp ((n_prims, 3)): (nodes (n, 16) float32, leaf entries int32)."""
    L = lib()
    flat = scene.flatten()
    cap = 4 * (flat.c.n_spheres + flat.c.n_polygons + flat.c.n_triangles) + 16
    nodes = np.zeros((cap, 16), dtype=np.float32)
    prims = np.zeros(cap, dtype=np.int32)
    n_nodes, n_prims = C.c_int(), C.c_int()
    v, vp = _disp(disp)
    rc = L.emu_swept_bvh(C.byref(flat.c), vp, nodes.ctypes.data, cap, prims.ctypes.data, cap, C.byref(n_nodes), C.byref(n_prims))
    if rc != 0:
        raise RuntimeError("emu_swept_bvh rc %d" % rc)
    return nodes[:n_nodes.value], prims[:n_prims.value]


def render(scene, width, height, disp, samples, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3, cull=True, threads=8,
           patch_rows=(0, -1), accel=False, glass_mode=None):
    """The FP32 motion frame (h, w, 3) float32 and the glass mode it was shaded in; disp: (n_prims, 3) by primitive id."""
    L = lib()
    L.emu_set_glass_mode(-1 if glass_mode is None else int(glass_mode))
    flat = scene.flatten()
    p = params(scene.camera, width, height, fov, max_depth, cull, patch_rows, accel)
    v, vp = _disp(disp)
    rgb = np.zeros((height, width, 3), dtype=np.float32)
    rc = L.emu_render_motion(C.byref(flat.c), C.byref(p), _basis(basis), C.byref(lens(aperture, focus, samples)), vp, rgb.ctypes.data,
                             threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "glass_mode": L.emu_last_glass_mode()}
