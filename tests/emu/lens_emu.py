"""ctypes binding of tests/emu/rm_lens_emu.cpp: rm_render_lens's per-ray kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from rusty_marcher_b200 import _abi

from . import emu

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_lens_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_lens_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_lens_offset.argtypes = [C.c_int, C.c_int, C.c_int, d]
        L.emu_lens_ray.argtypes = [C.POINTER(_abi.RmParams), d, C.POINTER(_abi.RmLens), C.c_int, C.c_int, C.c_int, C.c_int, d, d]
        L.emu_render_lens.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.POINTER(_abi.RmLens), C.c_void_p,
                                      C.c_int]
        _lib = L
    return _lib


def _basis(basis):
    return None if basis is None else (C.c_double * 9)(*[float(x) for x in np.asarray(basis).reshape(-1)])


def lens(aperture, focus, samples):
    ln = _abi.RmLens()
    ln.aperture, ln.focus, ln.samples = float(aperture), float(focus), int(samples)
    return ln


def params(camera, width, height, fov=1.5, max_depth=3, cull=True, patch_rows=(0, -1), accel=False):
    p = _abi.RmParams()
    p.width, p.height, p.fov = width, height, fov
    p.camera[:] = [float(c) for c in camera]
    p.max_depth, p.background, p.patch_size = max_depth, 0.1, 32
    p.patch_row_begin, p.patch_row_end = patch_rows
    p.cull_backfacing = int(cull)
    p.accel = int(accel)
    return p


def lens_offset(s, i, j):
    out = (C.c_double * 2)()
    lib().emu_lens_offset(s, i, j, out)
    return out[0], out[1]


def lens_ray(camera, width, height, fov, basis, aperture, focus, s, x, y, i, j):
    """(origin, direction) of sample (i, j) of pixel (x, y) from the library's rm::make_lens_camera and rm::lens_ray."""
    o, d = (C.c_double * 3)(), (C.c_double * 3)()
    p = params(camera, width, height, fov)
    lib().emu_lens_ray(C.byref(p), _basis(basis), C.byref(lens(aperture, focus, s)), x, y, i, j, o, d)
    return np.array(o[:]), np.array(d[:])


def render(scene, width, height, aperture, focus, samples, basis=None, fov=1.5, max_depth=3, cull=True, threads=8, patch_rows=(0, -1),
           accel=False, glass_mode=None):
    """The FP32 lens frame (h, w, 3) float32 and the glass mode it was shaded in."""
    L = lib()
    L.emu_set_glass_mode(-1 if glass_mode is None else int(glass_mode))
    flat = scene.flatten()
    p = params(scene.camera, width, height, fov, max_depth, cull, patch_rows, accel)
    rgb = np.zeros((height, width, 3), dtype=np.float32)
    rc = L.emu_render_lens(C.byref(flat.c), C.byref(p), _basis(basis), C.byref(lens(aperture, focus, samples)), rgb.ctypes.data, threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "glass_mode": L.emu_last_glass_mode()}
