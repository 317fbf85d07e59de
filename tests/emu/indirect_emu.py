"""ctypes binding of tests/emu/rm_indirect_emu.cpp: rm_render_indirect's per-ray kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from rusty_marcher_b200 import _abi

from . import emu
from .lens_emu import _basis, lens, params

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_indirect_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_indirect_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_diffuse_offset.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, d]
        L.emu_diffuse_ray.argtypes = [d, d, d, C.c_double, C.c_double, d, d]
        L.emu_render_indirect.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.POINTER(_abi.RmLens), C.c_void_p,
                                          C.c_int]
        L.emu_set_glass_mode.argtypes = [C.c_int]
        _lib = L
    return _lib


def _d(v):
    return (C.c_double * len(v))(*[float(x) for x in v])


def diffuse_offset(s, i, j, level):
    out = (C.c_double * 2)()
    lib().emu_diffuse_offset(s, i, j, level, out)
    return out[0], out[1]


def diffuse_ray(point, hit_normal, d, lx, ly):
    """(origin, direction) of the bounce at a hit of a ray of direction d, by rm::diffuse_origin / rm::diffuse_dir in f64."""
    o, r = (C.c_double * 3)(), (C.c_double * 3)()
    lib().emu_diffuse_ray(_d(point), _d(hit_normal), _d(d), float(lx), float(ly), o, r)
    return np.array(o[:]), np.array(r[:])


def render(scene, width, height, samples, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3, cull=True, threads=8,
           patch_rows=(0, -1), accel=False, glass_mode=None):
    """The FP32 indirect frame (h, w, 3) float32 and the glass mode it was shaded in."""
    L = lib()
    L.emu_set_glass_mode(-1 if glass_mode is None else int(glass_mode))
    flat = scene.flatten()
    p = params(scene.camera, width, height, fov, max_depth, cull, patch_rows, accel)
    rgb = np.zeros((height, width, 3), dtype=np.float32)
    rc = L.emu_render_indirect(C.byref(flat.c), C.byref(p), _basis(basis), C.byref(lens(aperture, focus, samples)), rgb.ctypes.data,
                               threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "glass_mode": L.emu_last_glass_mode()}
