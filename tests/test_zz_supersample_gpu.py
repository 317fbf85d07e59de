"""GPU part of the supersampled anti-aliasing tests (see tests/test_supersample.py): rm_render_supersampled against the
plain render it is defined by (bit for bit), against the oracle (the parity criteria of tests/parity.py), and its rows,
argument checks, retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi, workloads
from tests import parity
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), (O.Scene.create_default() if desc.get("default") else build_oracle_scene(desc))


def plain(rm, scene, w, h, rows=(0, -1), rgb8=False, depth=3):
    """rm_render's frame (float32) and, optionally, its 8-bit frame and maximum."""
    r = rm.create_renderer(1.5, h, w)
    r.max_depth = depth
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8) if rgb8 else None
    r.render(fb, scene, rgb8=b8, patch_rows=rows)
    return fb.buffer, b8, r.last_stats.max_value


def supersampled(rm, scene, w, h, s, rows=(0, -1), accel=False, depth=3, fill=0.):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    msg = r.render_supersampled(fb, scene, s, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


@pytest.mark.parametrize("name,w,h", [("demo", 800, 600), ("cornell_box", 640, 480)])
def test_one_sample_is_the_plain_render(rm_gpu, name, w, h):
    scene, _ = scenes(name)
    rgb, rgb8, mx = plain(rm_gpu, scene, w, h, rgb8=True)
    got, got8, st = supersampled(rm_gpu, scene, w, h, 1)
    assert np.array_equal(got.view(np.uint32), rgb.view(np.uint32))
    assert np.array_equal(got8, rgb8) and st.max_value == mx
    assert st.kernel_launches >= 4 and st.d2h_bytes == (h // 32) * 32 * w * 15 and st.ms_total >= st.ms_render > 0


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("name,w,h", [("demo", 800, 600), ("cornell_box", 640, 480)])
def test_frame_is_the_resolved_plain_render_of_the_larger_frame(rm_gpu, name, w, h, s):
    scene, _ = scenes(name)
    rows = (h // 32) * 32
    sub, _, _ = plain(rm_gpu, scene, s * w, s * h, rows=(0, s * (h // 32)))
    want = SS.resolve_f32(sub[:s * rows], s)
    got, got8, st = supersampled(rm_gpu, scene, w, h, s)
    assert np.array_equal(got[:rows].view(np.uint32), want.view(np.uint32))
    assert not got[rows:].any()
    assert st.max_value == float(want.max())
    assert np.array_equal(got8[:rows], SS.rgb8_of(want, want.max())) and not got8[rows:].any()


def check_parity(got, got8, ref, rows):
    a, b = got[:rows].astype(np.float64), ref[:rows]
    rel = (np.abs(a - b) / np.maximum(np.abs(b), 1e-12)).max(axis=2)
    frac = float((rel <= parity.REL_TOL).mean())
    assert frac >= parity.GOOD_FRACTION, "only %.5f of pixels within %g" % (frac, parity.REL_TOL)
    d = np.abs(got8[:rows].astype(np.int16) - parity.oracle_rgb8(ref)[:rows].astype(np.int16)).max(axis=2)
    frac8 = float((d <= 1).mean())
    assert frac8 >= parity.GOOD_FRACTION, "only %.5f of pixels within 1 LSB" % frac8
    return frac, frac8


@pytest.mark.parametrize("name,w,h,s", [("demo", 800, 600, 2), ("cornell_box", 640, 480, 2), ("dodecahedron", 640, 480, 2),
                                        ("demo", 800, 600, 3)])
def test_oracle_parity(rm_gpu, name, w, h, s):
    scene, osc = scenes(name)
    ref = SS.render_supersampled(osc, w, h, s)["rgb"]
    got, got8, _ = supersampled(rm_gpu, scene, w, h, s)
    print(name, s, check_parity(got, got8, ref, (h // 32) * 32))


def test_hierarchy_changes_no_pixel(rm_gpu):
    scene, _ = scenes("stress", n_spheres=64, grid=7)
    a, a8, sa = supersampled(rm_gpu, scene, 320, 224, 2, depth=6)
    b, b8, sb = supersampled(rm_gpu, scene, 320, 224, 2, depth=6, accel=True)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(a8, b8) and sa.max_value == sb.max_value
    assert a.any()


def test_rows_outside_the_call_are_left_untouched(rm_gpu):
    scene, _ = scenes("demo")
    full, _, _ = supersampled(rm_gpu, scene, 800, 600, 2, fill=np.nan)
    assert np.isnan(full[576:]).all() and np.isfinite(full[:576]).all()
    part, part8, _ = supersampled(rm_gpu, scene, 800, 600, 2, rows=(1, 3), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[96:]).all() and not part8[:32].any() and not part8[96:].any()
    assert np.array_equal(part[32:96], full[32:96]) and part8[32:96].any()


def test_argument_checks(rm_gpu):
    rm = rm_gpu
    scene, _ = scenes("demo")
    L = _abi.load()
    w, h = 128, 96
    p = rm.create_renderer(1.5, h, w).params(rm.create_frame_buffer(w, h), scene)
    hd = scene.device_handle()
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    assert L.rm_render_supersampled(hd, C.byref(p), 2, out.ctypes.data, out8.ctypes.data, None) == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()

    def call(samples=2, handle=hd, rgb=out.ctypes.data, rgb8=out8.ctypes.data, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        return L.rm_render_supersampled(handle, C.byref(q), samples, rgb, rgb8, None)

    assert call(samples=0) == -3 and call(samples=9) == -3
    assert call(patch_row_stride=2) == -3
    assert call(precision=_abi.RM_FP64) == -3
    assert call(handle=987654) == -3
    assert call(rgb=None, rgb8=None) == -3
    wide = np.zeros((64, 32768, 3), dtype=np.float32)
    assert call(width=32768, height=64, rgb=wide.ctypes.data, rgb8=None) == -4
    out[:] = 0
    out8[:] = 0
    st = _abi.RmStats()
    assert L.rm_render_supersampled(hd, C.byref(p), 2, out.ctypes.data, out8.ctypes.data, C.byref(st)) == 0
    assert np.array_equal(out, want) and np.array_equal(out8, want8) and st.max_value == float(want.max())


def test_a_retained_delivery_after_a_supersampled_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    supersampled call in between wrote the frame too, so the library must forget that delivery."""
    rm = rm_gpu
    w, h = 640, 480
    a, _ = scenes("cornell_box")
    b, _ = scenes("cornell_box")
    b.offset_camera((60., 25., 0.))
    fresh_a, _, _ = plain(rm, a, w, h)
    fresh_b, _, _ = plain(rm, b, w, h)
    r = rm.create_renderer(1.5, h, w)
    r.retained = True
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)
    r.render_supersampled(fb, b, 2)
    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the second camera lights tiles that are black in A's
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)
    assert not np.array_equal(fresh_a, fresh_b)


def test_headless_harness_saves_the_supersampled_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "aa.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "2", "--out", out], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_supersampled(fb, scene, 2, rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    assert subprocess.run([exe, "--samples", "9"], capture_output=True).returncode == 2
