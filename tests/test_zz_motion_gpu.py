"""GPU part of the motion-blur tests (see tests/test_motion.py): rm_render_motion against the oracle's motion frame
(tests/motion_ref.py) under the lens parity criterion, the routed cases against rm_render_lens (bit for bit), the kernel against
lens_kernel where the only mover can never be hit, the swept hierarchy against brute force, determinism, rows, the 8-bit frame,
argument checks, retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from rusty_marcher_b200.obj import Obj
from tests import lens_ref, motion_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def motion(rm, scene, w, h, disp, s, view=None, aperture=0., focus=1., accel=False, depth=3, rows=(0, -1), fill=0., cull=True):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel, r.cull_backfacing = depth, accel, cull
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_motion(fb, scene, disp, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


def lens(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3, cull=True):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel, r.cull_backfacing = depth, accel, cull
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    r.render_lens(fb, scene, aperture, focus, s, forward=fwd, up=up, rgb8=b8)
    return fb.buffer, b8, r.last_stats


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


def per_shape(scene, scale=1., seed=7):
    """one seeded displacement per shape, in multiples of 1/64 (exact in FP32)"""
    rng = np.random.default_rng(seed)
    return np.round(rng.uniform(-scale, scale, size=(len(scene.shapes), 3)) * 64.) / 64.


YAW30, PITCH = view_ref.VIEWS["yaw30"], view_ref.VIEWS["pitch-20"]
# (scene, width, height, max_depth, workload options, s, view, aperture, focus)
CASES = [("demo", 320, 256, 3, {}, 2, None, 0., 1.), ("demo", 320, 256, 3, {}, 4, None, 0., 1.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 2, None, 0., 1.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 4, None, 0., 1.),
         ("stress", 320, 192, 6, dict(n_spheres=256, grid=24), 2, None, 0., 1.),
         ("demo", 320, 256, 3, {}, 3, YAW30, 0., 1.), ("demo", 320, 256, 3, {}, 3, PITCH, 0.4, 12.)]


@pytest.mark.parametrize("c", CASES, ids=["%s-s%d-%s%s" % (c[0], c[5], "view" if c[6] else "none", "-lens" if c[7] else "") for c in CASES])
def test_motion_frames_meet_the_parity_criterion(rm_gpu, c):
    name, w, h, depth, kw, s, view, aperture, focus = c
    scene, oscene = scenes(name, **kw)
    v = per_shape(scene)
    basis = None if view is None else view_ref.numpy_basis(*view)
    ref = motion_ref.render(oscene, w, h, motion_ref.per_prim(scene, v), s, basis=basis, aperture=aperture, focus=focus, max_depth=depth)
    for accel in ([False, True] if name == "stress" else [False]):
        got, got8, st = motion(rm_gpu, scene, w, h, v, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth, cull=False)
        print(name, s, view is not None, accel, lens_ref.check_parity(got, got8, ref, (h // 32) * 32))
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        assert not same(got, lens(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth, cull=False)[0])


@pytest.mark.parametrize("kind", ["s1", "zero"])
@pytest.mark.parametrize("view", [None, YAW30], ids=["none", "yaw30"])
def test_routed_calls_are_the_lens_frame(rm_gpu, kind, view):
    scene, _ = scenes("stress", n_spheres=256, grid=24)
    s = 1 if kind == "s1" else 3
    v = (0.5, -0.25, 1.) if kind == "s1" else (0., 0., 0.)
    got, got8, st = motion(rm_gpu, scene, 320, 192, v, s, view=view, aperture=0.5, focus=100., depth=5)
    want, want8, st0 = lens(rm_gpu, scene, 320, 192, s, view=view, aperture=0.5, focus=100., depth=5)
    assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value and got.any()


MATTE = dict(diffusion=1., diffuse_color=(0.7, 0.6, 0.5), specular=0.3, specular_exponent=30., is_glass_like=False, reflection=0.,
             refractive_index=1.)


def unhittable_mover():
    """The stress scene plus a clockwise-projected quad and triangle that move (never hit, culled or not); the rest at rest."""
    desc = workloads.describe("stress", n_spheres=256, grid=24)
    desc["polygons"] = [([(-5., -5., -20.), (-5., 5., -20.), (5., 5., -20.), (5., -5., -20.)], MATTE),
                        ([(-8., -2., -25.), (-8., 4., -25.), (-2., 4., -25.)], MATTE)]
    scene = workloads.build_scene(desc)
    v = np.zeros((len(scene.shapes), 3))
    k = len(desc["spheres"])
    v[k] = v[k + 1] = (3.5, -1.25, 2.)
    return scene, v


@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("cull", [True, False])
def test_the_kernel_is_the_lens_kernel_where_the_mover_is_never_hit(rm_gpu, accel, cull):
    scene, v = unhittable_mover()
    got, got8, st = motion(rm_gpu, scene, 320, 192, v, 3, view=YAW30, accel=accel, depth=5, cull=cull)
    want, want8, _ = lens(rm_gpu, scene, 320, 192, 3, view=YAW30, accel=accel, depth=5, cull=cull)
    assert st.kernel_launches == 2                                 # the motion kernel ran (no routing)
    assert same(got, want) and np.array_equal(got8, want8) and got.any()


def nine_light_stress():
    desc = workloads.describe("stress", n_spheres=256, grid=24)
    lights = list(desc["lights"])
    while len(lights) < 9:
        k = len(lights)
        lights.append(((10. * k - 40., 30., 10.), (1., 0.8, 0.6), 0.3))
    desc["lights"] = lights
    return workloads.build_scene(desc)


@pytest.mark.parametrize("name", ["stress", "demo", "ngons", "stress9"])
def test_swept_hierarchy_and_repeat_change_no_pixel(rm_gpu, name):
    scene = nine_light_stress() if name == "stress9" else scenes(name)[0] if name == "demo" else \
        scenes(name, **(dict(n_spheres=256, grid=24) if name == "stress" else {}))[0]
    v = per_shape(scene, 2.)
    a, a8, sa = motion(rm_gpu, scene, 320, 192, v, 3, view=YAW30, depth=6)
    b, b8, sb = motion(rm_gpu, scene, 320, 192, v, 3, view=YAW30, depth=6, accel=True)
    c, c8, _ = motion(rm_gpu, scene, 320, 192, v, 3, view=YAW30, depth=6, accel=True)
    assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()
    assert same(b, c) and np.array_equal(b8, c8)
    d, _, _ = motion(rm_gpu, scene, 320, 192, v * 0.5, 3, view=YAW30, depth=6, accel=True)   # another motion: its own hierarchy
    e, _, _ = motion(rm_gpu, scene, 320, 192, v * 0.5, 3, view=YAW30, depth=6)
    assert same(d, e) and not same(d, a)


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("demo")
    v = per_shape(scene)
    full, full8, _ = motion(rm_gpu, scene, 320, 240, v, 3, fill=np.nan)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = motion(rm_gpu, scene, 320, 240, v, 3, rows=(1, 4), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, YAW30])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = motion(rm_gpu, scene, 320, 240, per_shape(scene), 2, view=view)
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
    n = scene.num_prims
    assert L.rm_scene_num_prims(hd) == n
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    v = np.ascontiguousarray(np.tile([0.5, 0.25, -0.5], (n + 1, 1)))

    def call(n_prims=n, samples=2, handle=hd, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, val in fields.items():
            setattr(q, k, val)
        m = _abi.RmMotion()
        m.n_prims, m.displacement, m.samples = n_prims, v.ctypes.data_as(C.POINTER(C.c_double)), samples
        return L.rm_render_motion(handle, C.byref(q), None, None, C.byref(m), out.ctypes.data, out8.ctypes.data, None)

    assert call() == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()
    assert call(n_prims=n + 1) == -3 and call(n_prims=n - 1) == -3
    assert call(handle=987654) == -3
    assert call(samples=9) == -3 and call(max_depth=0) == -3
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    m = _abi.RmMotion()
    m.n_prims, m.displacement, m.samples = n, v.ctypes.data_as(C.POINTER(C.c_double)), 8
    q = _abi.RmParams.from_buffer_copy(p)
    q.width, q.height = 16384, 64
    assert L.rm_render_motion(hd, C.byref(q), None, None, C.byref(m), wide.ctypes.data, None, None) == -4
    out[:] = 0
    out8[:] = 0
    assert call() == 0
    assert same(out, want) and np.array_equal(out8, want8)


def test_a_retained_delivery_after_a_motion_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    motion call in between wrote the frame too, so the library must forget that delivery."""
    rm = rm_gpu
    w, h = 640, 480
    a, _ = scenes("cornell_box")
    b, _ = scenes("demo")

    def fresh(scene):
        fb = rm.create_frame_buffer(w, h, dtype=np.float32)
        rm.create_renderer(1.5, h, w).render(fb, scene)
        return fb.buffer

    fresh_a = fresh(a)
    r = rm.create_renderer(1.5, h, w)
    r.retained = True
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)
    r.render_motion(fb, b, (1., 0., 0.), 2)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the demo frame lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)


def test_headless_harness_saves_the_motion_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "motion.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--move", "0,1.5,-0.5,0", "--aperture", "0.3",
                        "--focus", "12", "--look-at", "1,0,-10", "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    disp = np.zeros((len(scene.shapes), 3))
    disp[0] = (1.5, -0.5, 0.)
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_motion(fb, scene, disp, 3, forward=(1., 0., -10.), aperture=0.3, focus=12., rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    assert not isinstance(scene.shapes[0], Obj)
    for bad in (["--move", "0,1,0,0", "--roughness", "0.2"], ["--move", "0,1,0,0", "--light-radius", "1"],
                ["--move", "0,1,0,0", "--contrast", "0.1"], ["--move", "0,1,0,0", "--f64"], ["--move", "99,1,0,0"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
