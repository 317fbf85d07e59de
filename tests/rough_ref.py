"""The rough glass of rm_render_rough_glass (include/rm_b200.h RmRoughGlass) restated for the tests: the turned direction in
numpy, and the same plus the rough-glass frame over the CPU oracle (tests/rough_oracle.cpp).  Frames are checked with the lens
parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle
from rusty_marcher_b200.obj import Obj

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "rough_oracle.cpp")
LIB = os.path.join(HERE, "librough_oracle.so")
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
        L.orc_rough_dir.argtypes = [d, C.c_double, C.c_double, C.c_double, d]
        L.orc_rough_offset.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, d]
        L.orc_render_rough.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                       C.c_double, C.c_int, d, C.c_int, d, C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


def _d(v):
    return None if v is None else (C.c_double * len(v))(*[float(x) for x in v])


def numpy_rough_dir(rd, g, lx, ly):
    """rd turned by (lx, ly) with roughness g, operation for operation in numpy float64 scalars."""
    x, y, z = (np.float64(v) for v in rd)
    g, lx, ly = np.float64(g), np.float64(lx), np.float64(ly)
    if not g > 0. or (lx == 0. and ly == 0.):
        return np.array([x, y, z])
    sigma = np.copysign(np.float64(1.), z)
    alpha = np.float64(-1.) / (sigma + z)
    beta = (x * y) * alpha
    t1 = (np.float64(1.) + ((sigma * x) * x) * alpha, sigma * beta, -sigma * x)
    t2 = (beta, sigma + (y * y) * alpha, -y)
    v = [(x, y, z)[k] + g * ((lx * t1[k]) + (ly * t2[k])) for k in range(3)]
    norm = np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
    inv = np.float64(1.) / norm
    return np.array([v[0] * inv, v[1] * inv, v[2] * inv])


def oracle_rough_dir(rd, g, lx, ly):
    out = (C.c_double * 3)()
    lib().orc_rough_dir(_d(rd), float(g), float(lx), float(ly), out)
    return np.array(out[:])


def oracle_rough_offset(s, i, j, level):
    out = (C.c_double * 2)()
    lib().orc_rough_offset(s, i, j, level, out)
    return out[0], out[1]


def per_prim(scene, per_shape):
    """Per-shape values of a rusty_marcher_b200 Scene expanded to primitive ids (an Obj once per triangle)."""
    v = np.asarray(per_shape, dtype=np.float64)
    if v.ndim == 0:
        v = np.full(len(scene.shapes), float(v))
    return np.repeat(v, [s.triangles.shape[0] if isinstance(s, Obj) else 1 for s in scene.shapes])


def glass_like(scene):
    """is_glass_like by primitive id of a rusty_marcher_b200 Scene."""
    out = []
    for s in scene.shapes:
        if isinstance(s, Obj):
            out.extend(bool(f) for f in s.reflectances["is_glass_like"])
        else:
            out.append(bool(s.reflectance.is_glass_like))
    return np.array(out, dtype=bool)


def render(scene, width, height, roughness, samples, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3, threads=None,
           patch_rows=(0, -1)):
    """The oracle's rough-glass frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits}.
    roughness: one value per primitive id.  Rows outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    g = np.ascontiguousarray(roughness, dtype=np.float64)
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_rough(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]), int(patch_rows[1]),
                                _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture), float(focus), int(samples),
                                g.ctypes.data_as(C.POINTER(C.c_double)), g.shape[0], rgb.ctypes.data_as(C.POINTER(C.c_double)),
                                frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32 and samples in [1, 8]")
    return {"rgb": rgb, "fragile": frag}
