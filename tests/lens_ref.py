"""The thin-lens camera of rm_render_lens (include/rm_b200.h, RmLens) restated for the tests: the lens points in numpy, and
the sample rays and the lens frame over the CPU oracle (tests/lens_oracle.cpp); plus the lens parity criterion."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle
from tests import parity

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "lens_oracle.cpp")
LIB = os.path.join(HERE, "liblens_oracle.so")
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
        u8 = C.POINTER(C.c_uint8)
        L.orc_lens_offset.argtypes = [C.c_int, C.c_int, C.c_int, d]
        L.orc_lens_ray.argtypes = [d, C.c_int, C.c_int, C.c_double, d, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, d, d]
        L.orc_render_lens.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, d, C.c_double,
                                      C.c_double, C.c_int, d, d, u8, u8]
        _lib = L
    return _lib


def _d(v):
    return None if v is None else (C.c_double * len(v))(*[float(x) for x in v])


def numpy_lens_offset(s, i, j):
    """(lx, ly) of sample (i, j) of s x s, operation for operation in numpy float64 scalars."""
    a, b = (i + j) % s, j
    p = (np.float64(2.) * a + np.float64(1.)) / np.float64(s) - np.float64(1.)
    q = (np.float64(2.) * b + np.float64(1.)) / np.float64(s) - np.float64(1.)
    return p * np.sqrt(np.float64(1.) - (q * q) * np.float64(0.5)), q * np.sqrt(np.float64(1.) - (p * p) * np.float64(0.5))


def oracle_lens_offset(s, i, j):
    out = (C.c_double * 2)()
    lib().orc_lens_offset(s, i, j, out)
    return out[0], out[1]


def oracle_lens_ray(camera, width, height, fov, basis, aperture, focus, s, x, y, i, j):
    """(origin, direction) of sample (i, j) of pixel (x, y); basis: (3, 3) rows u, v, w, or None for the reference's camera."""
    o, d = (C.c_double * 3)(), (C.c_double * 3)()
    lib().orc_lens_ray(_d(camera), width, height, float(fov), _d(None if basis is None else np.asarray(basis).reshape(-1)),
                       float(aperture), float(focus), s, x, y, i, j, o, d)
    return np.array(o[:]), np.array(d[:])


def render(scene, width, height, aperture, focus, samples, basis=None, fov=1.5, max_depth=3, threads=None, patch_rows=(0, -1),
           want_samples=False):
    """The oracle's lens frame: {"rgb": (h, w, 3) f64 pixel means, "fragile": (h, w) OR of the samples' near-tie bits, and
    with want_samples "samples" (h, w, s*s, 3) and "sample_fragile" (h, w, s*s)}.  Rows outside the patch rows are zero."""
    if threads is None:
        threads = oracle.hardware_threads()
    ss = samples * samples
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    frag = np.zeros((height, width), dtype=np.uint8)
    smp = np.zeros((height, width, ss, 3), dtype=np.float64) if want_samples else None
    sfrag = np.zeros((height, width, ss), dtype=np.uint8) if want_samples else None
    u8 = C.POINTER(C.c_uint8)
    rc = lib().orc_render_lens(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]), int(patch_rows[1]),
                               _d(None if basis is None else np.asarray(basis).reshape(-1)), float(aperture), float(focus), int(samples),
                               rgb.ctypes.data_as(C.POINTER(C.c_double)),
                               smp.ctypes.data_as(C.POINTER(C.c_double)) if want_samples else None,
                               sfrag.ctypes.data_as(u8) if want_samples else None, frag.ctypes.data_as(u8))
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32 and samples in [1, 8]")
    out = {"rgb": rgb, "fragile": frag}
    if want_samples:
        out["samples"], out["sample_fragile"] = smp, sfrag
    return out


def check_parity(rgb, rgb8, ref, rows):
    """The lens parity criterion over the rendered rows: pixels with a near-tie in the primary query of any of their samples
    are left out (their share is returned); on the rest at least 99.9 % of the pixels are within 1e-4 relative of the f64
    mean, and the 8-bit frame within 1 LSB of the oracle's normalize + to_vec."""
    keep = (ref["fragile"][:rows] & 1) == 0
    a, b = rgb[:rows].astype(np.float64), ref["rgb"][:rows]
    rel = (np.abs(a - b) / np.maximum(np.abs(b), 1e-12)).max(axis=2)
    frac = float((rel[keep] <= parity.REL_TOL).mean()) if keep.any() else 1.
    assert frac >= parity.GOOD_FRACTION, "only %.5f of the non-fragile pixels within %g" % (frac, parity.REL_TOL)
    d = np.abs(rgb8[:rows].astype(np.int16) - parity.oracle_rgb8(ref["rgb"])[:rows].astype(np.int16)).max(axis=2)
    frac8 = float((d[keep] <= 1).mean()) if keep.any() else 1.
    assert frac8 >= parity.GOOD_FRACTION, "only %.5f of the non-fragile pixels within 1 LSB" % frac8
    return {"fragile_frac": float(1. - keep.mean()), "frac_within_tol": frac, "frac_within_1lsb": frac8, "max_rel": float(rel[keep].max()) if keep.any() else 0.}
