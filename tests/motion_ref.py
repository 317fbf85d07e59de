"""The motion blur of rm_render_motion (include/rm_b200.h RmMotion) restated for the tests: the sample times in numpy, and the
same plus the motion frame over the CPU oracle (tests/motion_oracle.cpp), whose scene is moved to each sample's time.  Frames
are checked with the lens parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle
from rusty_marcher_b200.obj import Obj

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "motion_oracle.cpp")
LIB = os.path.join(HERE, "libmotion_oracle.so")
DEPS = [SRC, os.path.join(HERE, "lens_oracle.cpp")] + [os.path.join(os.path.dirname(HERE), "oracle", f) for f in ("rm_oracle.cpp", "rm_oracle.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in DEPS):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-pthread", "-shared",
                            "-o", LIB, SRC], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.orc_motion_time.restype = C.c_double
        L.orc_motion_time.argtypes = [C.c_int, C.c_int, C.c_int]
        L.orc_render_motion.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                        C.c_double, C.c_int, d, C.c_int, d, C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


def _d(v):
    return None if v is None else (C.c_double * len(v))(*[float(x) for x in v])


def numpy_motion_time(s, i, j):
    """The time of sample (i, j) of s x s, operation for operation in numpy float64 scalars."""
    m = s * ((2 * i + j) % s) + (i + j) % s
    return (np.float64(m) + np.float64(0.5)) / np.float64(s * s) - np.float64(0.5)


def oracle_motion_time(s, i, j):
    return lib().orc_motion_time(s, i, j)


def per_prim(scene, per_shape):
    """Per-shape displacements (one 3-vector, or one per shape) of a rusty_marcher_b200 Scene expanded to primitive ids (an
    Obj once per triangle): (n_prims, 3) float64."""
    v = np.asarray(per_shape, dtype=np.float64)
    if v.shape == (3,):
        v = np.tile(v, (len(scene.shapes), 1))
    return np.ascontiguousarray(np.repeat(v, [s.triangles.shape[0] if isinstance(s, Obj) else 1 for s in scene.shapes], axis=0))


def render(scene, width, height, disp, samples, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3, threads=None,
           patch_rows=(0, -1)):
    """The oracle's motion frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits}.
    disp: (n_prims, 3) by primitive id.  Rows outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    v = np.ascontiguousarray(disp, dtype=np.float64).reshape(-1, 3)
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_motion(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]), int(patch_rows[1]),
                                 _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture), float(focus), int(samples),
                                 v.ctypes.data_as(C.POINTER(C.c_double)), v.shape[0], rgb.ctypes.data_as(C.POINTER(C.c_double)),
                                 frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32, samples in [1, 8], one displacement per primitive")
    return {"rgb": rgb, "fragile": frag}
