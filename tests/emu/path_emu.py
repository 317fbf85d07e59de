"""ctypes binding of tests/emu/rm_path_emu.cpp: rm_render_path's per-ray kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from rusty_marcher_b200 import _abi

from . import emu
from .lens_emu import _basis, lens, params

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_path_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_path_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_render_path.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.POINTER(_abi.RmLens), d, d,
                                      C.c_int, d, C.c_void_p, C.c_int]
        L.emu_set_glass_mode.argtypes = [C.c_int]
        _lib = L
    return _lib


def _arr(v, shape=None):
    if v is None:
        return None, None
    a = np.ascontiguousarray(v, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


def render(scene, width, height, samples, radii=None, roughness=None, disp=None, basis=None, aperture=0., focus=1., fov=1.5,
           max_depth=3, cull=True, threads=8, patch_rows=(0, -1), accel=False, glass_mode=None):
    """The FP32 path-traced frame (h, w, 3) float32 and the glass mode it was shaded in.  radii: one per light of the scene;
    roughness: one per primitive id; disp: (n_prims, 3) by primitive id; None: no such effect (disp given runs the motion
    code whatever its values)."""
    L = lib()
    L.emu_set_glass_mode(-1 if glass_mode is None else int(glass_mode))
    flat = scene.flatten()
    p = params(scene.camera, width, height, fov, max_depth, cull, patch_rows, accel)
    r, rp = _arr(radii)
    g, gp = _arr(roughness)
    v, vp = _arr(disp, (-1, 3))
    rgb = np.zeros((height, width, 3), dtype=np.float32)
    rc = L.emu_render_path(C.byref(flat.c), C.byref(p), _basis(basis), C.byref(lens(aperture, focus, samples)), rp, gp,
                           0 if g is None else g.shape[0], vp, rgb.ctypes.data, threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "glass_mode": L.emu_last_glass_mode()}
