"""GPU part of the rough-glass tests (see tests/test_rough.py): rm_render_rough_glass against the oracle's rough frame
(tests/rough_ref.py) under the lens parity criterion, the routed cases against rm_render_lens and rm_render_supersampled (bit
for bit), the kernel against lens_kernel where nothing can turn, the hierarchy, determinism, rows, the 8-bit frame, argument
checks, retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import lens_ref, rough_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def rough(rm, scene, w, h, roughness, s, view=None, aperture=0., focus=1., accel=False, depth=3, rows=(0, -1), fill=0.):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_rough_glass(fb, scene, roughness, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


def lens(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    r.render_lens(fb, scene, aperture, focus, s, forward=fwd, up=up, rgb8=b8)
    return fb.buffer, b8, r.last_stats


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


def glass_only(scene, g):
    """one roughness per shape: g on the glass-like spheres and polygons, 0 elsewhere (an Obj's first triangle decides)"""
    return [g if (bool(s.reflectances["is_glass_like"][0]) if hasattr(s, "reflectances") else s.reflectance.is_glass_like) else 0.
            for s in scene.shapes]


YAW30, PITCH = view_ref.VIEWS["yaw30"], view_ref.VIEWS["pitch-20"]
# (scene, width, height, max_depth, workload options, roughness, s, view, aperture, focus)
CASES = [("demo", 320, 256, 3, {}, 0.1, 2, None, 0., 1.), ("demo", 320, 256, 3, {}, 0.1, 4, None, 0., 1.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 0.2, 2, None, 0., 1.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 0.2, 4, None, 0., 1.),
         ("stress", 320, 192, 6, dict(n_spheres=256, grid=24), 0.05, 2, None, 0., 1.),
         ("demo", 320, 256, 3, {}, 0.1, 3, YAW30, 0., 1.), ("demo", 320, 256, 3, {}, 0.1, 3, PITCH, 0.4, 12.)]


@pytest.mark.parametrize("c", CASES, ids=["%s-s%d-%s%s" % (c[0], c[6], "view" if c[7] else "none", "-lens" if c[8] else "") for c in CASES])
def test_rough_frames_meet_the_parity_criterion(rm_gpu, c):
    name, w, h, depth, kw, g, s, view, aperture, focus = c
    scene, oscene = scenes(name, **kw)
    per_shape = glass_only(scene, g)
    basis = None if view is None else view_ref.numpy_basis(*view)
    ref = rough_ref.render(oscene, w, h, rough_ref.per_prim(scene, per_shape), s, basis=basis, aperture=aperture, focus=focus,
                           max_depth=depth)
    accels = [False, True] if name == "stress" else [False]
    for accel in accels:
        got, got8, st = rough(rm_gpu, scene, w, h, per_shape, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth)
        print(name, s, view is not None, accel, lens_ref.check_parity(got, got8, ref, (h // 32) * 32))
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        assert not same(got, lens(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth)[0])


@pytest.mark.parametrize("kind", ["s1", "zero", "opaque"])
@pytest.mark.parametrize("view", [None, YAW30], ids=["none", "yaw30"])
def test_routed_calls_are_the_lens_frame(rm_gpu, kind, view):
    scene, _ = scenes("stress", n_spheres=256, grid=24)
    s = 1 if kind == "s1" else 3
    g = 0.3 if kind == "s1" else 0. if kind == "zero" else [0. if v else 0.3 for v in glass_only(scene, 1.)]
    got, got8, st = rough(rm_gpu, scene, 320, 192, g, s, view=view, aperture=0.5, focus=100., depth=5)
    want, want8, st0 = lens(rm_gpu, scene, 320, 192, s, view=view, aperture=0.5, focus=100., depth=5)
    assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value and got.any()


def test_cornell_box_with_roughness_is_the_supersampled_frame(rm_gpu):
    scene, _ = scenes("cornell_box")
    got, got8, _ = rough(rm_gpu, scene, 320, 256, 0.3, 3)
    r = rm_gpu.create_renderer(1.5, 256, 320)
    fb = rm_gpu.create_frame_buffer(320, 256, dtype=np.float32)
    b8 = np.zeros((256, 320, 3), dtype=np.uint8)
    r.render_supersampled(fb, scene, 3, rgb8=b8)
    assert same(got, fb.buffer) and np.array_equal(got8, b8) and got.any()


def sealed_scene():
    """The demo scene plus a rough glass sphere sealed inside an opaque one: no ray reaches the glass."""
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    glass = dict(diffusion=0.1, diffuse_color=(1., 1., 1.), specular=0.5, specular_exponent=100., is_glass_like=True, reflection=0.1,
                 refractive_index=1.5)
    matte = dict(diffusion=1., diffuse_color=(0.7, 0.6, 0.5), specular=0.3, specular_exponent=30., is_glass_like=False, reflection=0.,
                 refractive_index=1.)
    desc["spheres"] = list(desc["spheres"]) + [((3., -2., -40.), 4., matte), ((3., -2., -40.), 1., glass)]
    scene = workloads.build_scene(desc)
    return scene, [0.] * (len(scene.shapes) - 1) + [0.4]


@pytest.mark.parametrize("accel", [False, True])
def test_the_kernel_is_the_lens_kernel_where_nothing_turns(rm_gpu, accel):
    scene, g = sealed_scene()
    got, got8, st = rough(rm_gpu, scene, 320, 192, g, 3, view=YAW30, accel=accel, depth=5)
    want, want8, _ = lens(rm_gpu, scene, 320, 192, 3, view=YAW30, accel=accel, depth=5)
    assert st.kernel_launches == 2                                 # the rough kernel ran (no routing)
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
def test_hierarchy_and_repeat_change_no_pixel(rm_gpu, name):
    scene = nine_light_stress() if name == "stress9" else scenes(name)[0] if name == "demo" else \
        scenes(name, **(dict(n_spheres=256, grid=24) if name == "stress" else {}))[0]
    a, a8, sa = rough(rm_gpu, scene, 320, 192, 0.2, 3, view=YAW30, depth=6)
    b, b8, sb = rough(rm_gpu, scene, 320, 192, 0.2, 3, view=YAW30, depth=6, accel=True)
    c, c8, _ = rough(rm_gpu, scene, 320, 192, 0.2, 3, view=YAW30, depth=6, accel=True)
    assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()
    assert same(b, c) and np.array_equal(b8, c8)


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("demo")
    full, full8, _ = rough(rm_gpu, scene, 320, 240, 0.15, 3, fill=np.nan)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = rough(rm_gpu, scene, 320, 240, 0.15, 3, rows=(1, 4), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, YAW30])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = rough(rm_gpu, scene, 320, 240, 0.15, 2, view=view)
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
    g = np.full(n + 1, 0.2)

    def call(n_prims=n, samples=2, handle=hd, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        r = _abi.RmRoughGlass()
        r.n_prims, r.roughness, r.samples = n_prims, g.ctypes.data_as(C.POINTER(C.c_double)), samples
        return L.rm_render_rough_glass(handle, C.byref(q), None, None, C.byref(r), out.ctypes.data, out8.ctypes.data, None)

    assert call() == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()
    assert call(n_prims=n + 1) == -3 and call(n_prims=n - 1) == -3
    assert call(handle=987654) == -3
    assert call(samples=9) == -3 and call(max_depth=0) == -3
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    r = _abi.RmRoughGlass()
    r.n_prims, r.roughness, r.samples = n, g.ctypes.data_as(C.POINTER(C.c_double)), 8
    q = _abi.RmParams.from_buffer_copy(p)
    q.width, q.height = 16384, 64
    assert L.rm_render_rough_glass(hd, C.byref(q), None, None, C.byref(r), wide.ctypes.data, None, None) == -4
    out[:] = 0
    out8[:] = 0
    assert call() == 0
    assert same(out, want) and np.array_equal(out8, want8)


def test_a_retained_delivery_after_a_rough_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    rough call in between wrote the frame too, so the library must forget that delivery."""
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
    r.render_rough_glass(fb, b, 0.2, 2)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the demo frame lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)


def test_headless_harness_saves_the_rough_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "rough.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--roughness", "0.2", "--aperture", "0.3",
                        "--focus", "12", "--look-at", "1,0,-10", "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_rough_glass(fb, scene, 0.2, 3, forward=(1., 0., -10.), aperture=0.3, focus=12., rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--roughness", "0.2", "--light-radius", "1"], ["--roughness", "0.2", "--contrast", "0.1"],
                ["--roughness", "0.2", "--f64"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
