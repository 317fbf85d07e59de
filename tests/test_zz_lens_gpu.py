"""GPU part of the depth-of-field tests (see tests/test_lens.py): rm_render_lens without aperture against
rm_render_supersampled and rm_render (bit for bit), with a lens against the oracle's lens frame (tests/lens_ref.py) under the
lens parity criterion, the hierarchy on against off, rows, the 8-bit frame, argument checks, retained-frame bookkeeping and
the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import lens_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def lens(rm, scene, w, h, aperture, focus, s, view=None, accel=False, depth=3, rows=(0, -1), fill=0.):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_lens(fb, scene, aperture, focus, s, forward=fwd, up=up, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


def supersampled(rm, scene, w, h, s, depth=3):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth = depth
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    r.render_supersampled(fb, scene, s, rgb8=b8)
    return fb.buffer, b8, r.last_stats


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


@pytest.mark.parametrize("s", [1, 2, 4])
def test_aperture_zero_is_the_supersampled_frame(rm_gpu, s):
    scene, _ = scenes("demo")
    want, want8, st0 = supersampled(rm_gpu, scene, 320, 256, s)
    got, got8, st = lens(rm_gpu, scene, 320, 256, 0., 12., s)
    assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value
    if s == 1:
        r = rm_gpu.create_renderer(1.5, 256, 320)
        fb = rm_gpu.create_frame_buffer(320, 256, dtype=np.float32)
        r.render(fb, scene)
        assert same(got, fb.buffer)


# (scene, width, height, max_depth, workload options, focus, aperture)
CASES = [("demo", 320, 256, 3, {}, 12., 0.4), ("cornell_box", 320, 256, 3, {}, 300., 8.),
         ("stress", 320, 192, 6, dict(n_spheres=256, grid=24), 120., 2.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 30., 0.6)]
VIEWS = {"none": None, "yaw30": view_ref.VIEWS["yaw30"], "pitch-20": view_ref.VIEWS["pitch-20"]}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw, focus, aperture = request.param
    scene, oscene = scenes(name, **kw)
    return name, w, h, depth, focus, aperture, scene, oscene


@pytest.mark.parametrize("s,view", [(2, "none"), (3, "yaw30"), (4, "none"), (2, "pitch-20")])
def test_lens_frames_meet_the_parity_criterion(rm_gpu, case, s, view):
    name, w, h, depth, focus, aperture, scene, oscene = case
    v = VIEWS[view]
    ref = lens_ref.render(oscene, w, h, aperture, focus, s, basis=None if v is None else view_ref.numpy_basis(*v), max_depth=depth)
    accels = [False, True] if name == "stress" else [False]
    for accel in accels:
        got, got8, st = lens(rm_gpu, scene, w, h, aperture, focus, s, view=v, accel=accel, depth=depth)
        print(name, s, view, accel, lens_ref.check_parity(got, got8, ref, (h // 32) * 32))
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        assert got.any() or (name == "cornell_box" and view == "yaw30")


@pytest.mark.parametrize("name,kw,focus,aperture", [("stress", dict(n_spheres=256, grid=24), 120., 2.), ("demo", {}, 12., 0.4),
                                                    ("ngons", {}, 30., 0.6)])
def test_hierarchy_changes_no_pixel(rm_gpu, name, kw, focus, aperture):
    scene, _ = scenes(name, **kw)
    a, a8, sa = lens(rm_gpu, scene, 320, 192, aperture, focus, 3, depth=6)
    b, b8, sb = lens(rm_gpu, scene, 320, 192, aperture, focus, 3, depth=6, accel=True)
    assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("demo")
    full, full8, _ = lens(rm_gpu, scene, 320, 240, 0.5, 12., 3, fill=np.nan)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = lens(rm_gpu, scene, 320, 240, 0.5, 12., 3, rows=(1, 4), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, view_ref.VIEWS["yaw30"]])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = lens(rm_gpu, scene, 320, 240, 0.5, 12., 2, view=view)
    rows = 224
    assert st.max_value == float(got[:rows].max()) > 0
    assert np.array_equal(got8[:rows], SS.rgb8_of(got[:rows], got[:rows].max())) and not got8[rows:].any()
    assert st.d2h_bytes == rows * 320 * 15


def test_argument_checks(rm_gpu):
    rm = rm_gpu
    scene, _ = scenes("demo")
    L = _abi.load()
    w, h = 128, 96
    p = rm.create_renderer(1.5, h, w).params(rm.create_frame_buffer(w, h), scene)
    hd = scene.device_handle()
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    ln = _abi.RmLens()
    ln.aperture, ln.focus, ln.samples = 0.5, 12., 2
    assert L.rm_render_lens(hd, C.byref(p), None, C.byref(ln), out.ctypes.data, out8.ctypes.data, None) == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()

    def call(handle=hd, rgb=out.ctypes.data, rgb8=out8.ctypes.data, view=None, lens_fields=(), **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        m = _abi.RmLens.from_buffer_copy(ln)
        for k, v in lens_fields:
            setattr(m, k, v)
        return L.rm_render_lens(handle, C.byref(q), view, C.byref(m), rgb, rgb8, None)

    assert call(lens_fields=[("samples", 0)]) == -3 and call(lens_fields=[("samples", 9)]) == -3
    assert call(lens_fields=[("aperture", -1.)]) == -3 and call(lens_fields=[("focus", 0.)]) == -3
    assert call(lens_fields=[("focus", float("nan"))]) == -3
    assert L.rm_render_lens(hd, C.byref(p), None, None, out.ctypes.data, None, None) == -3
    bad = rm.renderer._view((0., 1., 0.), (0., 1., 0.))
    assert call(view=C.byref(bad)) == -3
    assert call(patch_row_stride=2) == -3 and call(precision=_abi.RM_FP64) == -3 and call(max_depth=0) == -3
    assert call(handle=987654) == -3
    assert call(rgb=None, rgb8=None) == -3
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    assert call(width=16384, height=64, rgb=wide.ctypes.data, rgb8=None, lens_fields=[("samples", 8)]) == -4
    out[:] = 0
    out8[:] = 0
    st = _abi.RmStats()
    assert L.rm_render_lens(hd, C.byref(p), None, C.byref(ln), out.ctypes.data, out8.ctypes.data, C.byref(st)) == 0
    assert same(out, want) and np.array_equal(out8, want8) and st.max_value == float(want.max())


def test_a_retained_delivery_after_a_lens_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    lens call in between wrote the frame too, so the library must forget that delivery."""
    rm = rm_gpu
    w, h = 640, 480
    a, _ = scenes("cornell_box")
    b, _ = scenes("cornell_box")
    b.offset_camera((60., 25., 0.))

    def fresh(scene):
        fb = rm.create_frame_buffer(w, h, dtype=np.float32)
        rm.create_renderer(1.5, h, w).render(fb, scene)
        return fb.buffer

    fresh_a, fresh_b = fresh(a), fresh(b)
    r = rm.create_renderer(1.5, h, w)
    r.retained = True
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)
    r.render_lens(fb, b, 5., 300., 2)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the second camera lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)
    assert not np.array_equal(fresh_a, fresh_b)


def test_headless_harness_saves_the_lens_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "dof.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--aperture", "0.5", "--focus", "12",
                        "--look-at", "1,0,-10", "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_lens(fb, scene, 0.5, 12., 3, forward=(1., 0., -10.), rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--aperture", "0.5"], ["--aperture", "0.5", "--focus", "12", "--f64"],
                ["--aperture", "0.5", "--focus", "12", "--contrast", "0.1"], ["--aperture", "0.5", "--focus", "12", "--rows-f64"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
