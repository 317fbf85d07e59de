"""The diffuse interreflection of rm_render_indirect (include/rm_b200.h) restated for the tests: the strata and disc points in
Python, and the same plus the bounce direction and the indirect frame over the CPU oracle (tests/indirect_oracle.cpp).  Frames
are checked with the lens parity criterion (tests/lens_ref.py check_parity) unchanged."""
import ctypes as C
import math
import os
import subprocess

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "indirect_oracle.cpp")
LIB = os.path.join(HERE, "libindirect_oracle.so")
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
        L.orc_diffuse_offset.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, d]
        L.orc_diffuse_dir.argtypes = [d, C.c_double, C.c_double, d]
        L.orc_render_indirect.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                          C.c_double, C.c_int, d, C.POINTER(C.c_uint8)]
        _lib = L
    return _lib


def _d(v):
    return None if v is None else (C.c_double * len(v))(*[float(x) for x in v])


def stratum(s, i, j, level):
    return (2 * i + 3 * j + level) % s, (3 * i + 5 * j) % s


def python_diffuse_point(s, a, b):
    """The concentric map of the centre of stratum (a, b) of s x s, operation for operation in Python floats (math.cos and
    math.sin call the C library, as the library's host code does)."""
    p, q = (2. * a + 1.) / s - 1., (2. * b + 1.) / s - 1.
    if p == 0. and q == 0.:
        return 0., 0.
    if abs(p) > abs(q):
        r, phi = p, (math.pi / 4.) * (q / p)
    else:
        r, phi = q, math.pi / 2. - (math.pi / 4.) * (p / q)
    return r * math.cos(phi), r * math.sin(phi)


def python_diffuse_offset(s, i, j, level):
    return python_diffuse_point(s, *stratum(s, i, j, level))


def oracle_diffuse_offset(s, i, j, level):
    out = (C.c_double * 2)()
    lib().orc_diffuse_offset(s, i, j, level, out)
    return out[0], out[1]


def oracle_diffuse_dir(nf, lx, ly):
    out = (C.c_double * 3)()
    lib().orc_diffuse_dir(_d(nf), float(lx), float(ly), out)
    return np.array(out[:])


def render(scene, width, height, samples, basis=None, aperture=0., focus=1., fov=1.5, max_depth=3, threads=None, patch_rows=(0, -1)):
    """The oracle's indirect frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits}.
    Rows outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    rc = lib().orc_render_indirect(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]),
                                   int(patch_rows[1]), _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture),
                                   float(focus), int(samples), rgb.ctypes.data_as(C.POINTER(C.c_double)),
                                   frag.ctypes.data_as(C.POINTER(C.c_uint8)))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32 and samples in [1, 8]")
    return {"rgb": rgb, "fragile": frag}


# ---- scenes of the tests ----
def furnace_desc(rho):
    refl = dict(diffusion=1., diffuse_color=(rho, rho, rho), specular=0.5, specular_exponent=30., is_glass_like=False, reflection=0.,
                refractive_index=1.)
    return {"name": "furnace", "default": False, "spheres": [((0., 0., 0.), 100., refl)], "polygons": [], "meshes": [],
            "lights": [((0., 0., -50.), (0., 0., 0.), 1.)]}           # a black light adds exactly +0


def furnace_value(rho, depth, bg=0.1):
    return bg * sum(rho ** k for k in range(depth))


BLEED_CENTRE, BLEED_RADIUS = (0., 0., -24.), 3.


def bleed_desc():
    red = dict(diffusion=1., diffuse_color=(0.9, 0.05, 0.05), specular=0., specular_exponent=30., is_glass_like=False, reflection=0.,
               refractive_index=1.)
    white = dict(diffusion=1., diffuse_color=(0.9, 0.9, 0.9), specular=0., specular_exponent=30., is_glass_like=False, reflection=0.,
                 refractive_index=1.)
    wall = ([(-60., -60., -30.), (60., -60., -30.), (60., 60., -30.), (-60., 60., -30.)], white)       # CCW: normal +z
    return {"name": "bleed", "default": False, "spheres": [(BLEED_CENTRE, BLEED_RADIUS, red)], "polygons": [wall], "meshes": [],
            "lights": [((0., 0., 10.), (1., 1., 1.), 1.)]}


def anchor_desc(with_target=True, spheres=True):
    black = dict(diffusion=1., diffuse_color=(0., 0., 0.), specular=0.6, specular_exponent=30., is_glass_like=False, reflection=0.,
                 refractive_index=1.)
    glass = dict(diffusion=0.5, diffuse_color=(0.5, 0.7, 0.9), specular=0.5, specular_exponent=100., is_glass_like=True, reflection=0.1,
                 refractive_index=1.5)
    diffuse = dict(diffusion=1., diffuse_color=(0.9, 0.9, 0.9), specular=0., specular_exponent=30., is_glass_like=False, reflection=0.,
                   refractive_index=1.)
    floor = ([(-40., -8., -60.), (40., -8., -60.), (40., -8., 0.), (-40., -8., 0.)][::-1], black)
    back = ([(-40., -8., -40.), (40., -8., -40.), (40., 30., -40.), (-40., 30., -40.)], black)
    polygons = [floor, back]
    if with_target:
        # behind the camera, far below everything: no primary ray, no bounce (nothing else bounces) and no shadow ray (the
        # lights are above every surface) reaches it; wound clockwise as seen from the camera
        polygons.append(([(200., -300., 60.), (230., -330., 60.), (170., -330., 60.)], diffuse))
    sph = [((-4., 0., -20.), 3., black), ((5., 1., -25.), 4., glass)] if spheres else []
    return {"name": "anchor", "default": False, "spheres": sph, "polygons": polygons, "meshes": [],
            "lights": [((-10., 40., -10.), (1., 1., 1.), 1.), ((20., 30., 0.), (0.8, 0.6, 0.4), 0.9)]}
