"""The spherical area lights of rm_render_area_lights (include/rm_b200.h RmAreaLights) restated for the tests: the light frame
and the sample points in numpy, and the same plus the area-light frame over the CPU oracle (tests/area_oracle.cpp).  Frames
are checked with the lens parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "area_oracle.cpp")
LIB = os.path.join(HERE, "libarea_oracle.so")
ORACLE_SRC = [os.path.join(os.path.dirname(HERE), "oracle", f) for f in ("rm_oracle.cpp", "rm_oracle.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in [SRC] + ORACLE_SRC):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-pthread", "-shared",
                            "-o", LIB, SRC], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.orc_lens_offset_area.argtypes = [C.c_int, C.c_int, C.c_int, d]
        L.orc_light_frame.argtypes = [d, d, d]
        L.orc_light_sample.argtypes = [d, C.c_double, d, d, C.c_double, C.c_double, d]
        L.orc_render_area.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_int, C.c_int,
                                      d, C.POINTER(C.c_int32), C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


def _d(v):
    return (C.c_double * len(v))(*[float(x) for x in v])


def numpy_light_frame(m):
    """(t1, t2) of the unit vector m, operation for operation in numpy float64 scalars."""
    mx, my, mz = (np.float64(v) for v in m)
    sigma = np.copysign(np.float64(1.), mz)
    alpha = np.float64(-1.) / (sigma + mz)
    beta = (mx * my) * alpha
    return (np.array([np.float64(1.) + ((sigma * mx) * mx) * alpha, sigma * beta, -sigma * mx]),
            np.array([beta, sigma + (my * my) * alpha, -my]))


def numpy_light_sample(c, r, t1, t2, lx, ly):
    r, lx, ly = np.float64(r), np.float64(lx), np.float64(ly)
    return np.array([np.float64(c[k]) + r * ((lx * np.float64(t1[k])) + (ly * np.float64(t2[k]))) for k in range(3)])


def oracle_light_frame(m):
    t1, t2 = (C.c_double * 3)(), (C.c_double * 3)()
    lib().orc_light_frame(_d(m), t1, t2)
    return np.array(t1[:]), np.array(t2[:])


def oracle_light_sample(c, r, t1, t2, lx, ly):
    q = (C.c_double * 3)()
    lib().orc_light_sample(_d(c), float(r), _d(t1), _d(t2), float(lx), float(ly), q)
    return np.array(q[:])


def render(scene, width, height, radii, samples, fov=1.5, max_depth=3, threads=None, patch_rows=(0, -1)):
    """The oracle's area-light frame: {"rgb": (h, w, 3) f64, "prim_id": (h, w) int32, "fragile": (h, w) near-tie bits (bit 0:
    the primary query, bit 1: any decision, shadow rays included)}.  Rows outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    prim = np.full((height, width), -1, dtype=np.int32)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_area(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]), int(patch_rows[1]),
                               _d(radii), len(radii), int(samples), rgb.ctypes.data_as(C.POINTER(C.c_double)),
                               prim.ctypes.data_as(C.POINTER(C.c_int32)), frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32, samples in [1, 8], one radius per light")
    return {"rgb": rgb, "prim_id": prim, "fragile": frag}
