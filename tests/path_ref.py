"""The path-traced frame of rm_render_path (include/rm_b200.h) restated for the tests over the CPU oracle
(tests/path_oracle.cpp): the distributed frame of tests/distributed_oracle.cpp with rm_render_indirect's diffuse bounce.  Frames
are checked with the lens parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "path_oracle.cpp")
LIB = os.path.join(HERE, "libpath_oracle.so")
DEPS = [SRC] + [os.path.join(HERE, f) for f in ("distributed_oracle.cpp", "motion_oracle.cpp", "lens_oracle.cpp")] + \
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
        L.orc_render_path.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                      C.c_double, C.c_int, d, C.c_int, d, C.c_int, d, C.c_int, d, C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


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
    """The oracle's path-traced frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits}.
    radii: one per light; roughness: one per primitive id; disp: (n_prims, 3) by primitive id; None: no such effect.  Rows
    outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    r, rp, nr = _arr(radii)
    g, gp, ng = _arr(roughness)
    v, vp, nv = _arr(disp, (-1, 3))
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_path(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]), int(patch_rows[1]),
                               _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture), float(focus), int(samples),
                               rp, nr, gp, ng, vp, nv, rgb.ctypes.data_as(C.POINTER(C.c_double)), frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32, samples in [1, 8], one radius per light, one displacement "
                         "per primitive")
    return {"rgb": rgb, "fragile": frag}


# ---- scenes of the tests ----
GLASS = dict(diffusion=0.5, diffuse_color=(0.5, 0.7, 0.9), specular=0.5, specular_exponent=100., is_glass_like=True, reflection=0.1,
             refractive_index=1.5)


def with_inert_triangle(scene, g=0.3):
    """The scene plus, as its last shape, a glass-like triangle wound clockwise in the image plane: it never passes the
    reference's inside test (polygon.rs:83-91), so it is never hit and never shadows, and cull_backfacing drops it.  Returns
    the scene and the roughness by primitive id: g on the triangle, which makes rough glass an active effect, 0 elsewhere."""
    from rusty_marcher_b200 import polygon
    from rusty_marcher_b200.geometry import Vec3f
    from rusty_marcher_b200.shapes import Reflectance
    r = GLASS
    refl = Reflectance(r["diffusion"], Vec3f(*r["diffuse_color"]), r["specular"], r["specular_exponent"], r["is_glass_like"],
                       r["reflection"], r["refractive_index"])
    scene.shapes.append(polygon.ConvexPolygon.create([Vec3f(-8., -2., -25.), Vec3f(-8., 4., -25.), Vec3f(-2., 4., -25.)], refl))
    g_by_prim = np.zeros(scene.num_prims)
    g_by_prim[-1] = g
    return scene, g_by_prim
