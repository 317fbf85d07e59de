"""Distributed ray tracing of rm_render_distributed (include/rm_b200.h) restated for the tests: rule 4's light stratum
(area_offset) in numpy, and the same plus the distributed frame over the CPU oracle (tests/distributed_oracle.cpp), whose scene
is moved to each sample's time, whose glass turns as rough glass's and whose area lights are one point per sample ray.  Frames
are checked with the lens parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "distributed_oracle.cpp")
LIB = os.path.join(HERE, "libdistributed_oracle.so")
DEPS = [SRC, os.path.join(HERE, "motion_oracle.cpp"), os.path.join(HERE, "lens_oracle.cpp")] + \
    [os.path.join(os.path.dirname(HERE), "oracle", f) for f in ("rm_oracle.cpp", "rm_oracle.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in DEPS):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-pthread", "-shared",
                            "-o", LIB, SRC], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.orc_area_offset.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, d]
        L.orc_render_distributed.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                             C.c_double, C.c_int, d, C.c_int, d, C.c_int, d, C.c_int, d, C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


def numpy_area_offset(s, i, j, level):
    """(lx, ly) of rule 4's stratum ((i + 2j + L) mod s, (i + 3j) mod s), operation for operation in numpy float64 scalars."""
    a, b = (i + 2 * j + level) % s, (i + 3 * j) % s
    f = np.float64
    p = (f(2.) * f(a) + f(1.)) / f(s) - f(1.)
    q = (f(2.) * f(b) + f(1.)) / f(s) - f(1.)
    return p * np.sqrt(f(1.) - (q * q) * f(0.5)), q * np.sqrt(f(1.) - (p * p) * f(0.5))


def oracle_area_offset(s, i, j, level):
    out = (C.c_double * 2)()
    lib().orc_area_offset(s, i, j, level, out)
    return out[0], out[1]


def _d(v):
    return None if v is None else (C.c_double * len(v))(*[float(x) for x in v])


def _arr(v, shape=None):
    if v is None:
        return None, None, 0
    a = np.ascontiguousarray(v, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a, a.ctypes.data_as(C.POINTER(C.c_double)), a.shape[0]


def render(scene, width, height, samples, radii=None, roughness=None, disp=None, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3,
           threads=None, patch_rows=(0, -1)):
    """The oracle's distributed frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits}.
    radii: one per light; roughness: one per primitive id; disp: (n_prims, 3) by primitive id; None: no such effect.  Rows
    outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    r, rp, nr = _arr(radii)
    g, gp, ng = _arr(roughness)
    v, vp, nv = _arr(disp, (-1, 3))
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_distributed(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]),
                                      int(patch_rows[1]), _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture),
                                      float(focus), int(samples), rp, nr, gp, ng, vp, nv, rgb.ctypes.data_as(C.POINTER(C.c_double)),
                                      frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32, samples in [1, 8], one radius per light, one displacement "
                         "per primitive")
    return {"rgb": rgb, "fragile": frag}
