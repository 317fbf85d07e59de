"""GPU part of the adaptive anti-aliasing tests (see tests/test_adaptive.py): rm_render_adaptive against the two calls it is
defined by -- rm_render (P, with its primary ids) and rm_render_supersampled (S) -- bit for bit, its mask against
tests/adaptive_ref.py, and its rows, argument checks, retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import adaptive_ref as AR
from tests import supersample_ref as SS

pytestmark = pytest.mark.gpu
INF = float("inf")


def scene_of(name, **kw):
    return workloads.build_scene(workloads.describe(name, **kw))


def plain(rm, scene, w, h, accel=False, depth=3):
    """rm_render's frame (float32), primary ids, 8-bit frame and maximum."""
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    ids = np.full((h, w), -1, dtype=np.int32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    r.render(fb, scene, prim_id=ids, rgb8=b8)
    return fb.buffer, ids, b8, r.last_stats.max_value


def supersampled(rm, scene, w, h, s, accel=False, depth=3):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    r.render_supersampled(fb, scene, s, rgb8=b8)
    return fb.buffer, b8, r.last_stats.max_value


def adaptive(rm, scene, w, h, s, contrast, rows=(0, -1), accel=False, depth=3, fill=0.):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    mask = np.zeros((h, w), dtype=np.uint8)
    msg = r.render_adaptive(fb, scene, s, contrast, rgb8=b8, mask=mask, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, mask, r.last_stats


def same(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


@pytest.mark.parametrize("contrast", [0., 0.1, INF, -1.])
@pytest.mark.parametrize("name,w,h", [("demo", 800, 600), ("cornell_box", 640, 480)])
def test_one_sample_is_the_plain_render(rm_gpu, name, w, h, contrast):
    scene = scene_of(name)
    rgb, ids, rgb8, mx = plain(rm_gpu, scene, w, h)
    got, got8, mask, st = adaptive(rm_gpu, scene, w, h, 1, contrast)
    assert same(got, rgb) and np.array_equal(got8, rgb8) and st.max_value == mx
    assert np.array_equal(mask, AR.mark(rgb, ids, contrast))
    assert st.kernel_launches >= 6 and st.d2h_bytes == (h // 32) * 32 * w * 16 and st.ms_total >= st.ms_render > 0


def check_refine_all(rm, scene, w, h, s, accel=False, depth=3):
    want, want8, mx = supersampled(rm, scene, w, h, s, accel=accel, depth=depth)
    got, got8, mask, st = adaptive(rm, scene, w, h, s, -1., accel=accel, depth=depth)
    rows = (h // 32) * 32
    assert same(got, want), "%d of %d pixels differ" % ((got[:rows] != want[:rows]).any(axis=2).sum(), rows * w)
    assert np.array_equal(got8, want8) and st.max_value == mx
    assert mask[:rows].all() and not mask[rows:].any()
    return got


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("name,w,h", [("demo", 800, 600), ("cornell_box", 640, 480), ("dodecahedron", 640, 480)])
def test_refining_every_pixel_is_the_supersampled_frame(rm_gpu, name, w, h, s):
    """Every sub-pixel value the sub-pixel kernel traces from the list equals K1's value for that pixel of the s x frame."""
    check_refine_all(rm_gpu, scene_of(name), w, h, s)


@pytest.mark.parametrize("accel", [False, True])
def test_refining_every_pixel_is_the_supersampled_frame_stress(rm_gpu, accel):
    got = check_refine_all(rm_gpu, scene_of("stress", n_spheres=64, grid=7), 320, 224, 2, accel=accel, depth=6)
    assert got.any()


@pytest.mark.parametrize("contrast", [0.05, 0.1, INF])
@pytest.mark.parametrize("s", [2, 4])
@pytest.mark.parametrize("name,w,h", [("demo", 800, 600), ("cornell_box", 640, 480)])
def test_frame_is_the_supersampled_frame_where_the_mask_is_set(rm_gpu, name, w, h, s, contrast):
    scene = scene_of(name)
    rgb, ids, _, _ = plain(rm_gpu, scene, w, h)
    sup, _, _ = supersampled(rm_gpu, scene, w, h, s)
    got, got8, mask, st = adaptive(rm_gpu, scene, w, h, s, contrast)
    rows = (h // 32) * 32
    want_mask = AR.mark(rgb, ids, contrast)
    assert np.array_equal(mask, want_mask)
    assert 0 < mask.sum() < rows * w
    want = AR.compose(want_mask, sup, rgb)
    assert same(got, want)
    assert st.max_value == float(want[:rows].max())
    assert np.array_equal(got8[:rows], SS.rgb8_of(want[:rows], want[:rows].max())) and not got8[rows:].any()
    print(name, s, contrast, "refined %.4f" % (mask.sum() / (rows * w)))


def test_hierarchy_changes_no_pixel(rm_gpu):
    scene = scene_of("stress", n_spheres=64, grid=7)
    a, a8, ma, sa = adaptive(rm_gpu, scene, 320, 224, 2, 0.1, depth=6)
    b, b8, mb, sb = adaptive(rm_gpu, scene, 320, 224, 2, 0.1, depth=6, accel=True)
    assert same(a, b) and np.array_equal(a8, b8) and np.array_equal(ma, mb) and sa.max_value == sb.max_value
    assert a.any() and 0 < ma.sum() < 224 * 320


def test_rows_outside_the_call_are_left_untouched(rm_gpu):
    scene = scene_of("demo")
    full, full8, fmask, _ = adaptive(rm_gpu, scene, 800, 600, 2, 0.1, fill=np.nan)
    assert np.isnan(full[576:]).all() and np.isfinite(full[:576]).all() and not fmask[576:].any()
    part, part8, pmask, _ = adaptive(rm_gpu, scene, 800, 600, 2, 0.1, rows=(1, 3), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[96:]).all()
    assert not part8[:32].any() and not part8[96:].any() and not pmask[:32].any() and not pmask[96:].any()
    assert same(part[32:96], full[32:96]) and part8[32:96].any()
    assert np.array_equal(pmask[32:96], fmask[32:96])
    assert fmask[[32, 95]].any()                                # rows whose mask needs the halo rows 31 and 96


def test_a_call_that_refines_nothing_is_the_plain_render(rm_gpu):
    rm = rm_gpu
    # a wall across the whole view: one primitive id in every pixel, so +inf (geometric edges only) refines nothing
    wall = dict(diffusion=1., diffuse_color=(0.8, 0.6, 0.4), specular=1., specular_exponent=30., is_glass_like=False,
                reflection=0.95, refractive_index=1.)
    desc = {"name": "wall", "default": False, "spheres": [], "meshes": [],
            "polygons": [([(-1000., -1000., -20.), (1000., -1000., -20.), (1000., 1000., -20.), (-1000., 1000., -20.)], wall)],
            "lights": [((5., 5., 0.), (1., 1., 1.), 1.)]}
    for scene in (workloads.build_scene(desc), rm.Scene()):    # ... and an empty scene, at any contrast
        rgb, ids, rgb8, mx = plain(rm, scene, 640, 480)
        got, got8, mask, st = adaptive(rm, scene, 640, 480, 4, INF if scene.shapes else 0.1)
        assert not mask.any() and same(got, rgb) and np.array_equal(got8, rgb8) and st.max_value == mx
    assert rgb8.sum() == 0 and ids.max() == -1


def test_argument_checks(rm_gpu):
    rm = rm_gpu
    scene = scene_of("demo")
    L = _abi.load()
    w, h = 128, 96
    p = rm.create_renderer(1.5, h, w).params(rm.create_frame_buffer(w, h), scene)
    hd = scene.device_handle()
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    mask = np.zeros((h, w), dtype=np.uint8)
    assert L.rm_render_adaptive(hd, C.byref(p), 2, 0.1, out.ctypes.data, out8.ctypes.data, mask.ctypes.data, None) == 0
    want, want8, wmask = out.copy(), out8.copy(), mask.copy()
    assert want.any() and wmask.any()

    def call(samples=2, contrast=0.1, handle=hd, rgb=out.ctypes.data, rgb8=out8.ctypes.data, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        return L.rm_render_adaptive(handle, C.byref(q), samples, contrast, rgb, rgb8, mask.ctypes.data, None)

    assert call(samples=0) == -3 and call(samples=9) == -3
    assert call(contrast=float("nan")) == -3
    assert call(patch_row_stride=2) == -3
    assert call(precision=_abi.RM_FP64) == -3
    assert call(max_depth=0) == -3
    assert call(handle=987654) == -3
    assert call(rgb=None, rgb8=None) == -3
    wide = np.zeros((64, 32768, 3), dtype=np.float32)
    assert call(width=32768, height=64, rgb=wide.ctypes.data, rgb8=None) == -4
    out[:] = 0
    out8[:] = 0
    mask[:] = 0
    st = _abi.RmStats()
    assert L.rm_render_adaptive(hd, C.byref(p), 2, 0.1, out.ctypes.data, out8.ctypes.data, mask.ctypes.data, C.byref(st)) == 0
    assert same(out, want) and np.array_equal(out8, want8) and np.array_equal(mask, wmask) and st.max_value == float(want.max())


def test_a_retained_delivery_after_an_adaptive_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    adaptive call in between wrote the frame too, so the library must forget that delivery."""
    rm = rm_gpu
    w, h = 640, 480
    a = scene_of("cornell_box")
    b = scene_of("cornell_box")
    b.offset_camera((60., 25., 0.))
    fresh_a, _, _, _ = plain(rm, a, w, h)
    fresh_b, _, _, _ = plain(rm, b, w, h)
    r = rm.create_renderer(1.5, h, w)
    r.retained = True
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)
    r.render_adaptive(fb, b, 2, 0.1)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the second camera lights tiles that are black in A's
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)
    assert not np.array_equal(fresh_a, fresh_b)


def test_headless_harness_saves_the_adaptive_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "aa.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "2", "--contrast", "0.1", "--out", out],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    mask = np.zeros((h, w), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_adaptive(fb, scene, 2, 0.1, rgb8=rgb8, mask=mask)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    assert ("%d of %d pixels refined" % (int(mask.sum()), w * h)) in r.stdout
    assert subprocess.run([exe, "--contrast", "nan"], capture_output=True).returncode == 2
