"""ctypes binding of tests/emu/rm_view_emu.cpp: rm_render_view's kernel code compiled for the host."""
import ctypes as C
import os
import subprocess

import numpy as np

from rusty_marcher_b200 import _abi

from . import emu

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librm_view_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        srcs = [os.path.join(HERE, "rm_view_emu.cpp"), os.path.join(HERE, "rm_emu.cpp")] + [
            os.path.join(emu.ROOT, "rusty_marcher_b200", "csrc", f) for f in
            ("rm_trace.cuh", "rm_fast.cuh", "rm_math.cuh", "rm_scene.cpp", "rm_scene.h", "rm_host.cpp", "rm_bvh.cuh", "rm_bvh.cpp")]
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-pthread",
                            "-o", LIB, srcs[0]], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.emu_render_fast_view.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.c_void_p, C.c_void_p, C.c_int]
        L.emu_render_f64_view.argtypes = [C.POINTER(_abi.RmFlatScene), C.POINTER(_abi.RmParams), d, C.c_void_p, C.c_void_p,
                                          C.POINTER(_abi.RmStats), C.c_int]
        L.emu_view_basis.argtypes = [C.POINTER(_abi.RmView), d]
        _lib = L
    return _lib


def basis(forward, up):
    """(3, 3) rows u, v, w from the library's host code (rm::view_basis), or None for an invalid view."""
    v = _abi.RmView()
    v.forward[:] = [float(x) for x in forward]
    v.up[:] = [float(x) for x in up]
    out = np.zeros(9, dtype=np.float64)
    if lib().emu_view_basis(C.byref(v), out.ctypes.data_as(C.POINTER(C.c_double))) != 0:
        return None
    return out.reshape(3, 3)


def render(scene, width, height, view, precision="fast", fov=1.5, max_depth=3, cull=True, threads=8, patch_rows=(0, -1),
           strip_bound=True, accel=False):
    """precision "fast": the FP32 production path under the view; "f64": the FP64 validation kernel's code."""
    b = basis(*view)
    if b is None:
        raise ValueError("invalid view %r" % (view,))
    L = lib()
    L.emu_set_strip_bound(int(strip_bound))
    L.emu_set_glass_mode(-1)
    flat = scene.flatten()
    p = _abi.RmParams()
    p.width, p.height, p.fov = width, height, fov
    p.camera[:] = list(scene.camera)
    p.max_depth, p.background, p.patch_size = max_depth, 0.1, 32
    p.patch_row_begin, p.patch_row_end = patch_rows
    p.cull_backfacing = int(cull)
    p.accel = int(accel)
    dt = np.float32 if precision == "fast" else np.float64
    rgb = np.zeros((height, width, 3), dtype=dt)
    ids = np.full((height, width), -1, dtype=np.int32)
    bp = b.reshape(-1).ctypes.data_as(C.POINTER(C.c_double))
    st = _abi.RmStats()
    if precision == "fast":
        rc = L.emu_render_fast_view(C.byref(flat.c), C.byref(p), bp, rgb.ctypes.data, ids.ctypes.data, threads)
    else:
        rc = L.emu_render_f64_view(C.byref(flat.c), C.byref(p), bp, rgb.ctypes.data, ids.ctypes.data, C.byref(st), threads)
    if rc != 0:
        raise RuntimeError("emu rc %d" % rc)
    return {"rgb": rgb, "prim_id": ids, "counters": st.counters() if precision != "fast" else None}
