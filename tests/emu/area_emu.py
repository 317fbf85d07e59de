"""ctypes binding of tests/emu/rm_area_emu.cpp: rm_render_area_lights's per-pixel kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from . import emu
from .lens_emu import params

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_area_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_area_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_light_frame.argtypes = [d, d, d]
        L.emu_light_sample.argtypes = [d, C.c_double, d, d, C.c_double, C.c_double, d]
        L.emu_render_area.argtypes = [C.c_void_p, C.c_void_p, d, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.emu_set_glass_mode.argtypes = [C.c_int]
        _lib = L
    return _lib


def _d(v):
    return (C.c_double * len(v))(*[float(x) for x in v])


def light_frame(m):
    t1, t2 = (C.c_double * 3)(), (C.c_double * 3)()
    lib().emu_light_frame(_d(m), t1, t2)
    return np.array(t1[:]), np.array(t2[:])


def light_sample(c, r, t1, t2, lx, ly):
    q = (C.c_double * 3)()
    lib().emu_light_sample(_d(c), float(r), _d(t1), _d(t2), float(lx), float(ly), q)
    return np.array(q[:])


def render(scene, width, height, radii, samples, fov=1.5, max_depth=3, cull=True, threads=8, patch_rows=(0, -1), accel=False):
    """The FP32 area-light frame {"rgb": (h, w, 3) float32, "prim_id": (h, w) int32, "glass_mode": int}."""
    L = lib()
    L.emu_set_glass_mode(-1)
    flat = scene.flatten()
    p = params(scene.camera, width, height, fov, max_depth, cull, patch_rows, accel)
    rgb = np.zeros((height, width, 3), dtype=np.float32)
    prim = np.full((height, width), -2, dtype=np.int32)
    rc = L.emu_render_area(C.addressof(flat.c), C.addressof(p), _d(radii), int(samples), rgb.ctypes.data, prim.ctypes.data, threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "prim_id": prim, "glass_mode": L.emu_last_glass_mode()}
