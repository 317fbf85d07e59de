"""Adaptive anti-aliasing (rm_render_adaptive, include/rm_b200.h) restated for the tests.

The mode has no reference behaviour; it is defined through two frames: P, the plain 1x frame with its primary ids, and S,
the supersampled frame (tests/supersample_ref.py).  `mark` is the normative refinement mask over P restated in numpy with
float32 operations, `compose` picks S where the mask is set and P elsewhere, and `render_adaptive` is the definition over
the f64 oracle."""
import numpy as np

from oracle import oracle as O
from tests import supersample_ref as SS


def call_rows(h, patch_rows=(0, -1)):
    """Pixel rows [r0, r1) of a call over patch rows (begin, end); end = -1 (or past the frame) is floor(H/32)."""
    b, e = patch_rows[0], patch_rows[1]
    if e < 0 or e > h // 32:
        e = h // 32
    b = min(max(b, 0), e)
    return 32 * b, 32 * e


def mark(rgb, ids, contrast, rows=None):
    """The refinement mask, (H, W) uint8, 1 = refined, over the pixel rows `rows` = (r0, r1) (default: all of [0, R)), zero
    elsewhere.  rgb: the 1x frame (H, W, 3), ids: its primary ids (H, W); only their rows [0, R), R = 32 floor(H/32), are
    read.  contrast < 0 refines every pixel; otherwise a pixel is refined when one of its 8 neighbours in [0, W) x [0, R)
    has another id or, for some channel, fabsf(a - b) > k * (a + b) with k = float32(contrast), all in float32."""
    h, w = ids.shape
    R = 32 * (h // 32)
    r0, r1 = (0, R) if rows is None else rows
    out = np.zeros((h, w), dtype=np.uint8)
    if contrast < 0:
        out[r0:r1] = 1
        return out
    P = np.asarray(rgb, dtype=np.float32)[:R]
    ident = np.asarray(ids)[:R]
    k = np.float32(contrast)
    ref = np.zeros((R, w), dtype=bool)
    with np.errstate(invalid="ignore", over="ignore"):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dy == 0 and dx == 0:
                    continue
                py, px = slice(max(0, -dy), R - max(0, dy)), slice(max(0, -dx), w - max(0, dx))
                qy, qx = slice(max(0, dy), R + min(0, dy)), slice(max(0, dx), w + min(0, dx))
                a, b = P[py, px], P[qy, qx]
                ref[py, px] |= (ident[py, px] != ident[qy, qx]) | (np.abs(a - b) > k * (a + b)).any(axis=2)
    out[r0:r1] = ref[r0:r1]
    return out


def compose(mask, supersampled, plain):
    """The frame: the supersampled pixel where the mask is set, the plain one elsewhere."""
    return np.where(mask[..., None] != 0, supersampled, plain)


def render_adaptive(scene, w, h, s, contrast, patch_rows=(0, -1)):
    """The definition over the oracle: P over the call's rows plus one patch row of halo on either side (f64), the mask of
    its float32 values, S from SS.render_supersampled.  Rows outside the call are zero.  Returns {"rgb", "mask"}."""
    r0, r1 = call_rows(h, patch_rows)
    rgb = np.zeros((h, w, 3), dtype=np.float64)
    m = np.zeros((h, w), dtype=np.uint8)
    if r1 > r0:
        b, e = r0 // 32, r1 // 32
        p = O.render(scene, w, h, patch_rows=(max(b - 1, 0), min(e + 1, h // 32)), want_fragile=False, want_counters=False)
        m = mark(p["rgb"].astype(np.float32), p["prim_id"], contrast, (r0, r1))
        sup = SS.render_supersampled(scene, w, h, s, patch_rows=(b, e))["rgb"]
        rgb[r0:r1] = compose(m, sup, p["rgb"])[r0:r1]
    return {"rgb": rgb, "mask": m}
