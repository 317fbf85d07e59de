"""The camera orientation of rm_render_view (include/rm_b200.h, RmView) restated for the tests: the basis in numpy and
over the CPU oracle (tests/view_oracle.cpp), and oracle.render with the primary rays turned by it."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "view_oracle.cpp")
LIB = os.path.join(HERE, "libview_oracle.so")
ORACLE_SRC = [os.path.join(os.path.dirname(HERE), "oracle", f) for f in ("rm_oracle.cpp", "rm_oracle.h")]
_lib = None

# the five views of the tests: (forward, up)
YAW30 = ((-np.sin(np.radians(30.)), 0., -np.cos(np.radians(30.))), (0., 1., 0.))
PITCH_M20 = ((0., -np.sin(np.radians(20.)), -np.cos(np.radians(20.))), (0., 1., 0.))
ROLL90 = ((0., 0., -1.), (1., 0., 0.))
FORWARD_X = ((1., 0., 0.), (0., 1., 0.))
DOWN = ((0., -1., 0.), (0., 0., -1.))
VIEWS = {"yaw30": YAW30, "pitch-20": PITCH_M20, "roll90": ROLL90, "forward+x": FORWARD_X, "down": DOWN}
IDENTITY = ((0., 0., -1.), (0., 1., 0.))


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(s) for s in [SRC] + ORACLE_SRC):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-pthread", "-shared",
                            "-o", LIB, SRC], check=True)
        L = C.CDLL(LIB)
        d = C.POINTER(C.c_double)
        L.orc_view_basis.argtypes = [d, d, d]
        L.orc_render_view.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, d,
                                      d, C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.POINTER(oracle.Counters)]
        L.orc_last_degenerate_hits.restype = C.c_uint64
        _lib = L
    return _lib


def _d(v, n):
    return (C.c_double * n)(*[float(x) for x in v])


def oracle_basis(forward, up):
    """(3, 3) rows u, v, w from the oracle's geometry.rs restatement, or None for an invalid view."""
    out = (C.c_double * 9)()
    if lib().orc_view_basis(_d(forward, 3), _d(up, 3), out) != 0:
        return None
    return np.array(out[:], dtype=np.float64).reshape(3, 3)


def numpy_basis(forward, up):
    """The definition, operation for operation in numpy float64 scalars (no contraction), or None for an invalid view."""
    f = [np.float64(x) for x in forward]
    up = [np.float64(x) for x in up]
    if not all(np.isfinite(x) for x in f + up):
        return None
    if f[0] * f[0] + f[1] * f[1] + f[2] * f[2] == 0.:
        return None

    def normalized(a):
        s = np.float64(1.) / np.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
        return [a[0] * s, a[1] * s, a[2] * s]

    def cross(a, b):
        return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]

    w = normalized([-f[0], -f[1], -f[2]])
    c = cross(up, w)
    if c[0] * c[0] + c[1] * c[1] + c[2] * c[2] <= np.float64(1e-20) * (up[0] * up[0] + up[1] * up[1] + up[2] * up[2]):
        return None
    u = normalized(c)
    return np.array([u, cross(w, u), w], dtype=np.float64)


def render(scene, width, height, view=None, fov=1.5, max_depth=3, threads=None, patch_rows=(0, -1), patch_stride=1,
           want_ids=True, want_fragile=True, want_counters=True):
    """oracle.render with the camera turned to view = (forward, up); view=None is oracle.render itself."""
    if view is None:
        return oracle.render(scene, width, height, fov=fov, max_depth=max_depth, threads=threads, patch_rows=patch_rows,
                             patch_stride=patch_stride, want_ids=want_ids, want_fragile=want_fragile, want_counters=want_counters)
    basis = oracle_basis(*view)
    if basis is None:
        raise ValueError("invalid view %r" % (view,))
    if threads is None:
        threads = oracle.hardware_threads()
    rgb = np.zeros((height, width, 3), dtype=np.float64)
    ids = np.full((height, width), -1, dtype=np.int32) if want_ids else None
    frag = np.zeros((height, width), dtype=np.uint8) if want_fragile else None
    cnt = oracle.Counters() if want_counters else None
    rc = lib().orc_render_view(scene._h, width, height, float(fov), int(max_depth), int(threads), int(patch_rows[0]),
                               int(patch_rows[1]), int(patch_stride), _d(basis.reshape(-1), 9),
                               rgb.ctypes.data_as(C.POINTER(C.c_double)),
                               ids.ctypes.data_as(C.POINTER(C.c_int32)) if want_ids else None,
                               frag.ctypes.data_as(C.POINTER(C.c_uint8)) if want_fragile else None,
                               C.byref(cnt) if want_counters else None)
    if rc != 0:
        raise ValueError("oracle: width must be a positive multiple of 32 (renderer.rs:107)")
    return {"rgb": rgb, "prim_id": ids, "fragile": frag, "counters": cnt.as_dict() if want_counters else None,
            "degenerate_hits": int(lib().orc_last_degenerate_hits())}
