"""Supersampled anti-aliasing (rm_render_supersampled, include/rm_b200.h) restated for the tests.

The mode has no reference behaviour; it is defined through the reference's own frame: the frame at s*W x s*H, box-filtered
down to W x H.  `render_supersampled` is that definition over the f64 oracle, `resolve_f32` the normative FP32 order of
the library's resolve, and `rgb8_of` the library's normalize + to_vec of a float32 frame by a given maximum."""
import numpy as np

from oracle import oracle as O


def resolve(sub, s, dtype):
    """Box mean of every s x s block of `sub` ((s*R, s*W, 3) -> (R, W, 3)) in the normative order: acc = 0; for i in [0, s):
    for j in [0, s): acc += v[i][j]; out = acc / (s*s), every operation rounded to `dtype`."""
    acc = np.zeros((sub.shape[0] // s, sub.shape[1] // s, 3), dtype=dtype)
    for i in range(s):
        for j in range(s):
            acc = acc + sub[i::s, j::s].astype(dtype)
    return acc / dtype(s * s)


def resolve_f32(sub, s):
    return resolve(np.asarray(sub, dtype=np.float32), s, np.float32)


def render_supersampled(scene, w, h, s, patch_rows=(0, -1), **kw):
    """The oracle's frame at (s*w, s*h) over patch rows [s*b, s*e), box-filtered in f64 in the normative order.  Rows
    outside [32 b, 32 e) are zero.  Returns {"rgb": (h, w, 3) float64}."""
    b, e = patch_rows[0], patch_rows[1]
    if e < 0 or e > h // 32:
        e = h // 32
    b = min(b, e)
    kw.setdefault("want_ids", False)
    kw.setdefault("want_fragile", False)
    kw.setdefault("want_counters", False)
    rgb = np.zeros((h, w, 3), dtype=np.float64)
    if e > b:
        sub = O.render(scene, s * w, s * h, patch_rows=(s * b, s * e), **kw)["rgb"][s * 32 * b:s * 32 * e]
        rgb[32 * b:32 * e] = resolve(sub, s, np.float64)
    return {"rgb": rgb}


def rgb8_of(rgb, mx):
    """normalize + to_vec of a float32 frame by the maximum `mx` (framebuffer.rs:40-82, as the tone-map kernel does it)."""
    mx = np.float32(mx)
    inv = np.float32(1) / mx if mx > 0 else np.float32(1)
    return (np.float32(255) * np.clip(rgb * inv, np.float32(0), np.float32(1))).astype(np.uint8)
