"""GPU part of the soft-shadow tests (see tests/test_area.py): rm_render_area_lights against the oracle's area frame
(tests/area_ref.py) under the lens parity criterion, its primary ids and misses against rm_render, s = 1 and zero radii
against rm_render bit for bit, the hierarchy on against off and reproducibility, rows, the 8-bit frame, argument checks,
retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import area_ref, lens_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene
from tests.test_kernel_emulation import _with_lights

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def area(rm, scene, w, h, radii, s, accel=False, depth=3, rows=(0, -1), fill=0.):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    ids = np.full((h, w), -7, dtype=np.int32)
    msg = r.render_area_lights(fb, scene, radii, s, prim_id=ids, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, ids, r.last_stats


def plain(rm, scene, w, h, accel=False, depth=3):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    ids = np.full((h, w), -7, dtype=np.int32)
    r.render(fb, scene, prim_id=ids, rgb8=b8)
    return fb.buffer, b8, ids, r.last_stats


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


RADII = (0., 3.)                                                # the light at the camera stays a point, the other is a sphere
# (scene, width, height, max_depth, workload options)
CASES = [("demo", 320, 256, 3, {}), ("cornell_box", 320, 256, 3, {}), ("stress", 320, 192, 6, dict(n_spheres=256, grid=24)),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40))]


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw = request.param
    scene, oscene = scenes(name, **kw)
    return name, w, h, depth, scene, oscene


@pytest.mark.parametrize("s", [2, 4])
def test_area_frames_meet_the_parity_criterion(rm_gpu, case, s):
    name, w, h, depth, scene, oscene = case
    ref = area_ref.render(oscene, w, h, RADII, s, max_depth=depth)
    want, want8, want_ids, _ = plain(rm_gpu, scene, w, h, depth=depth)
    for accel in ([False, True] if name == "stress" else [False]):
        got, got8, ids, st = area(rm_gpu, scene, w, h, RADII, s, accel=accel, depth=depth)
        print(name, s, accel, lens_ref.check_parity(got, got8, ref, (h // 32) * 32))
        assert st.kernel_launches == 3 and st.ms_total >= st.ms_render > 0
        assert np.array_equal(ids, want_ids)                     # primary visibility is rm_render's
        miss = want_ids < 0
        assert not got[miss].any() and not want[miss].any()      # black exactly where rm_render's misses are
        assert (got[~miss].max(axis=1) > 0).all()
        assert not same(got, want)


@pytest.mark.parametrize("radii,s", [((0., 3.), 1), ((0., 0.), 2), ((0., 0.), 4), ((5., 2.), 1)])
def test_one_sample_and_zero_radii_are_rm_renders_frame(rm_gpu, radii, s):
    scene, _ = scenes("demo")
    want, want8, want_ids, st0 = plain(rm_gpu, scene, 320, 256)
    got, got8, ids, st = area(rm_gpu, scene, 320, 256, radii, s)
    assert same(got, want) and np.array_equal(got8, want8) and np.array_equal(ids, want_ids) and st.max_value == st0.max_value


def _glass_stress():
    return workloads.build_scene(workloads.describe("stress", n_spheres=256, grid=24))


def _nine_lights():
    scene = workloads.build_scene(_with_lights(workloads.describe("stress", n_spheres=512, grid=32), 9))
    scene.offset_camera((7.5, -3.25, 20.0))
    return scene


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("which", ["glass_stress", "demo", "ngons", "nine_lights"])
def test_hierarchy_changes_no_pixel_and_frames_repeat(rm_gpu, which, s):
    scene = {"glass_stress": _glass_stress, "demo": lambda: scenes("demo")[0], "ngons": lambda: scenes("ngons")[0],
             "nine_lights": _nine_lights}[which]()
    radii = [0.5 + 0.5 * k for k in range(len(scene.lights))]
    radii[0] = 0.
    a = area(rm_gpu, scene, 320, 192, radii, s, depth=6)
    b = area(rm_gpu, scene, 320, 192, radii, s, depth=6, accel=True)
    c = area(rm_gpu, scene, 320, 192, radii, s, depth=6, accel=True)
    d = area(rm_gpu, scene, 320, 192, radii, s, depth=6)
    for x in (b, c, d):
        assert same(a[0], x[0]) and np.array_equal(a[1], x[1]) and np.array_equal(a[2], x[2]) and a[3].max_value == x[3].max_value
    assert a[0].any()


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("demo")
    full, full8, ids, _ = area(rm_gpu, scene, 320, 240, RADII, 3, fill=np.nan)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all() and (ids[224:] == -7).all()
    part, part8, pids, _ = area(rm_gpu, scene, 320, 240, RADII, 3, rows=(1, 4), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert (pids[:32] == -7).all() and (pids[128:] == -7).all() and np.array_equal(pids[32:128], ids[32:128])
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu):
    scene, _ = scenes("demo")
    got, got8, _, st = area(rm_gpu, scene, 320, 240, RADII, 2)
    rows = 224
    assert st.max_value == float(got[:rows].max()) > 0
    assert np.array_equal(got8[:rows], SS.rgb8_of(got[:rows], got[:rows].max())) and not got8[rows:].any()
    assert st.d2h_bytes == rows * 320 * 19


def test_argument_checks(rm_gpu):
    rm = rm_gpu
    scene, _ = scenes("demo")
    L = _abi.load()
    w, h = 128, 96
    p = rm.create_renderer(1.5, h, w).params(rm.create_frame_buffer(w, h), scene)
    hd = scene.device_handle()
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    radius = (C.c_double * 3)(0., 3., 1.)
    al = _abi.RmAreaLights()
    al.n_lights, al.radius, al.samples = 2, C.cast(radius, C.POINTER(C.c_double)), 2
    assert L.rm_render_area_lights(hd, C.byref(p), C.byref(al), out.ctypes.data, None, out8.ctypes.data, None) == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()

    def call(handle=hd, rgb=out.ctypes.data, rgb8=out8.ctypes.data, light_fields=(), **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        m = _abi.RmAreaLights.from_buffer_copy(al)
        for k, v in light_fields:
            setattr(m, k, v)
        return L.rm_render_area_lights(handle, C.byref(q), C.byref(m), rgb, None, rgb8, None)

    assert call(light_fields=[("samples", 0)]) == -3 and call(light_fields=[("samples", 9)]) == -3
    assert call(light_fields=[("n_lights", 1)]) == -3 and call(light_fields=[("n_lights", 3)]) == -3    # the scene has 2
    assert call(light_fields=[("radius", None)]) == -3
    radius[1] = -1.
    assert call() == -3
    radius[1] = float("nan")
    assert call() == -3
    radius[1] = 3.
    assert L.rm_render_area_lights(hd, C.byref(p), None, out.ctypes.data, None, None, None) == -3
    assert call(patch_row_stride=2) == -3 and call(precision=_abi.RM_FP64) == -3 and call(max_depth=0) == -3
    assert call(handle=987654) == -3
    assert call(rgb=None, rgb8=None) == -3
    out[:] = 0
    out8[:] = 0
    st = _abi.RmStats()
    assert L.rm_render_area_lights(hd, C.byref(p), C.byref(al), out.ctypes.data, None, out8.ctypes.data, C.byref(st)) == 0
    assert same(out, want) and np.array_equal(out8, want8) and st.max_value == float(want.max())


def test_a_retained_delivery_after_an_area_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    area-light call in between wrote the frame too, so the library must forget that delivery."""
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
    r.render_area_lights(fb, b, (0., 5.), 2)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the second camera lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)
    assert not np.array_equal(fresh_a, fresh_b)


def test_headless_harness_saves_the_area_light_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "soft.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--light-radius", "0,2.5", "--accel",
                        "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_area_lights(fb, scene, (0., 2.5), 3, rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--light-radius", "1", "--f64"], ["--light-radius", "1", "--contrast", "0.1"], ["--light-radius", "1", "--rows-f64"],
                ["--light-radius", "1", "--look-at", "0,0,-1"], ["--light-radius", "1", "--aperture", "0.5", "--focus", "12"],
                ["--light-radius", "1,2,3"], ["--light-radius", "x"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
