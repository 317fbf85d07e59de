"""GPU part of the path-traced frame tests (see tests/test_path.py): rm_render_path against the oracle's path-traced frame
(tests/path_ref.py) under the lens parity criterion, the three routed cases against rm_render_distributed and rm_render_indirect
(bit for bit), the inert-effect and never-hit anchors, the furnace's closed form, the hierarchy, determinism, rows, the 8-bit
frame, argument checks, retained-frame bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import indirect_ref, lens_ref, path_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene
from tests.test_distributed import area_radii

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _renderer(rm, w, h, depth, accel, cull):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel, r.cull_backfacing = depth, accel, cull
    return r


def path(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3, rows=(0, -1), fill=0., cull=True, **e):
    r = _renderer(rm, w, h, depth, accel, cull)
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_path(fb, scene, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8, patch_rows=rows, **e)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


def distributed(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3, cull=True, **e):
    r = _renderer(rm, w, h, depth, accel, cull)
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    r.render_distributed(fb, scene, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8, **e)
    return fb.buffer, b8, r.last_stats


def indirect(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3, cull=True):
    r = _renderer(rm, w, h, depth, accel, cull)
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    r.render_indirect(fb, scene, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8)
    return fb.buffer, b8, r.last_stats


def kernels_run(fn):
    """Names of the CUDA kernels that ran during fn(), recorded by torch.profiler (CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type.name == "CUDA"}
    names |= {k.name for e in prof.events() for k in getattr(e, "kernels", [])}
    return out, names


def ran(names, kernel):
    return any(kernel in n for n in names)


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


def effects(scene, which, g=0.1, r=3.):
    e = {}
    if "area" in which:
        e["light_radii"] = area_radii(scene, r)
    if "rough" in which:
        e["roughness"] = _rough_by_shape(scene, g)
    if "motion" in which:
        e["displacement"] = _disp_by_shape(scene)
    return e


def _rough_by_shape(scene, g):
    """g on every glass-like sphere and polygon, 0 elsewhere: one roughness per shape, as render_path takes it."""
    from rusty_marcher_b200.obj import Obj
    return np.array([0. if isinstance(s, Obj) or not s.reflectance.is_glass_like else g for s in scene.shapes])


def _disp_by_shape(scene, scale=1., seed=7):
    """One displacement per shape, seeded, in multiples of 1/64 (exact in FP32), up to `scale` per component."""
    rng = np.random.default_rng(seed)
    return np.round(rng.uniform(-scale, scale, size=(len(scene.shapes), 3)) * 64.) / 64.


def _by_prim(scene, e):
    """The oracle's per-primitive arrays of the Python call's per-shape effects."""
    from rusty_marcher_b200.renderer import _displacement_by_prim, _roughness_by_prim
    out = {}
    if "light_radii" in e:
        out["radii"] = e["light_radii"]
    if "roughness" in e:
        out["roughness"] = _roughness_by_prim(scene, e["roughness"])
    if "displacement" in e:
        out["disp"] = _displacement_by_prim(scene, e["displacement"])
    return out


YAW30, PITCH = view_ref.VIEWS["yaw30"], view_ref.VIEWS["pitch-20"]
# (scene, width, height, max_depth, workload options, s, view, aperture, focus, effects)
CASES = [("demo", 320, 256, 3, {}, 2, None, 0., 1., "area"), ("demo", 320, 256, 4, {}, 4, YAW30, 0.4, 12., "area+rough+motion"),
         ("cornell_box", 320, 256, 3, {}, 2, None, 0., 1., "area+motion"),
         ("cornell_box", 320, 256, 4, {}, 3, YAW30, 0., 1., "area+rough+motion"),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 2, None, 0., 1., "rough+motion"),
         ("stress", 320, 192, 4, dict(n_spheres=256, grid=24), 2, None, 0., 1., "area+rough+motion"),
         ("demo", 320, 256, 3, {}, 3, PITCH, 0.4, 12., "motion")]


@pytest.mark.parametrize("c", CASES, ids=["%s-s%d-%s%s-%s" % (c[0], c[5], "view" if c[6] else "none", "-lens" if c[7] else "", c[9])
                                          for c in CASES])
def test_path_frames_meet_the_parity_criterion(rm_gpu, c):
    name, w, h, depth, kw, s, view, aperture, focus, which = c
    scene, oscene = scenes(name, **kw)
    e = effects(scene, which)
    basis = None if view is None else view_ref.numpy_basis(*view)
    ref = path_ref.render(oscene, w, h, s, basis=basis, aperture=aperture, focus=focus, max_depth=depth, **_by_prim(scene, e))
    accels = [False, True] if name in ("stress", "cornell_box") else [False]
    for accel in accels:
        (got, got8, st), names = kernels_run(lambda: path(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel,
                                                          depth=depth, **e))
        assert ran(names, "path_kernel"), names
        r = lens_ref.check_parity(got, got8, ref, (h // 32) * 32)
        print(name, s, which, view is not None, accel, r)
        assert r["fragile_frac"] < 0.2, r
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        want = distributed(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth, **e)[0]
        assert not same(got, want)


# ---- routing: each routed case is the routed call's frame bit for bit ----
@pytest.mark.parametrize("kind", ["depth1", "no-bounce", "s1", "no-effect"])
def test_routed_calls_are_the_routed_frame(rm_gpu, kind):
    scene, depth, s = scenes("stress", n_spheres=256, grid=24)[0], 4, 3
    if kind == "depth1":
        depth = 1
    elif kind == "no-bounce":
        scene = workloads.build_scene(indirect_ref.anchor_desc(with_target=False))
    elif kind == "s1":
        s = 1
    e = effects(scene, "rough" if kind == "no-effect" else "area+rough+motion", g=0. if kind == "no-effect" else 0.1)
    kw = dict(view=YAW30, aperture=0.5, focus=30., depth=depth)
    (got, got8, st), names = kernels_run(lambda: path(rm_gpu, scene, 320, 192, s, **kw, **e))
    assert not ran(names, "path_kernel"), names
    if kind in ("depth1", "no-bounce"):
        assert ran(names, "distributed_kernel") or kind == "depth1" and ran(names, "lens_kernel"), names
        want, want8, st0 = distributed(rm_gpu, scene, 320, 192, s, **kw, **e)
    else:
        assert ran(names, "indirect_kernel"), names
        want, want8, st0 = indirect(rm_gpu, scene, 320, 192, s, **kw)
    assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value and got.any()


# ---- the inert-effect anchor: active rough glass that is never hit leaves rm_render_indirect's frame ----
@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("name", ["stress", "cornell_box"])
def test_the_kernel_is_the_indirect_kernel_where_the_effects_are_inert(rm_gpu, accel, cull, name):
    scene, g = path_ref.with_inert_triangle(scenes(name, **(dict(n_spheres=256, grid=24) if name == "stress" else {}))[0])
    rough = np.zeros(len(scene.shapes))
    rough[-1] = g[-1]
    kw = dict(view=YAW30, aperture=0.3, focus=12., accel=accel, depth=4, cull=cull)
    (got, got8, st), names = kernels_run(lambda: path(rm_gpu, scene, 320, 192, 3, roughness=rough, **kw))
    assert ran(names, "path_kernel") and not ran(names, "indirect_kernel"), names
    want, want8, _ = indirect(rm_gpu, scene, 320, 192, 3, **kw)
    assert same(got, want) and np.array_equal(got8, want8) and got.any()


# ---- the never-hit anchor: black opaque surfaces and one diffuse triangle no ray reaches leave rm_render_distributed's ----
@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("spheres", [True, False], ids=["spheres", "planes"])
def test_the_kernel_is_the_distributed_kernel_where_nothing_bounces(rm_gpu, accel, cull, spheres):
    scene = workloads.build_scene(indirect_ref.anchor_desc(spheres=spheres))
    e = dict(light_radii=area_radii(scene, 2.), roughness=_rough_by_shape(scene, 0.2))
    v = np.zeros((len(scene.shapes), 3))
    if spheres:
        v[0], v[1] = (0.5, -0.25, 0.75), (-0.75, 0.5, 0.25)
    e["displacement"] = v
    kw = dict(aperture=0.3, focus=20., accel=accel, depth=4, cull=cull)
    (got, got8, st), names = kernels_run(lambda: path(rm_gpu, scene, 320, 192, 3, **kw, **e))
    assert ran(names, "path_kernel") and not ran(names, "distributed_kernel"), names
    want, want8, _ = distributed(rm_gpu, scene, 320, 192, 3, **kw, **e)
    assert same(got, want) and np.array_equal(got8, want8) and got.any()


@pytest.mark.parametrize("depth", [2, 3, 5])
def test_furnace_closed_form(rm_gpu, depth):
    rho = 0.6
    scene = workloads.build_scene(indirect_ref.furnace_desc(rho))
    for accel in (False, True):
        (got, _, st), names = kernels_run(lambda: path(rm_gpu, scene, 256, 192, 3, depth=depth, accel=accel, light_radii=[5.],
                                                       displacement=[3., -2., 1.5]))
        assert ran(names, "path_kernel"), names
        assert np.abs(got[:192].astype(np.float64) / indirect_ref.furnace_value(rho, depth) - 1.).max() <= 1e-6


def nine_light_stress():
    desc = workloads.describe("stress", n_spheres=256, grid=24)
    lights = list(desc["lights"])
    while len(lights) < 9:
        k = len(lights)
        lights.append(((10. * k - 40., 30., 10.), (1., 0.8, 0.6), 0.3))
    desc["lights"] = lights
    return workloads.build_scene(desc)


@pytest.mark.parametrize("name", ["stress", "demo", "cornell_box", "ngons", "stress9"])
def test_hierarchy_and_repeat_change_no_pixel(rm_gpu, name):
    scene = nine_light_stress() if name == "stress9" else \
        scenes(name, **(dict(n_spheres=256, grid=24) if name == "stress" else dict(n_spheres=12, n_polygons=40) if name == "ngons" else {}))[0]
    e = effects(scene, "area+rough+motion", r=2.)
    a, a8, sa = path(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5, **e)
    b, b8, sb = path(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5, accel=True, **e)
    c, c8, _ = path(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5, accel=True, **e)
    assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()
    assert same(b, c) and np.array_equal(b8, c8)


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("cornell_box")
    e = effects(scene, "area+motion")
    full, full8, _ = path(rm_gpu, scene, 320, 240, 3, fill=np.nan, **e)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = path(rm_gpu, scene, 320, 240, 3, rows=(1, 4), fill=np.nan, **e)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, YAW30])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = path(rm_gpu, scene, 320, 240, 2, view=view, **effects(scene, "area+rough+motion"))
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
    radii = np.full(len(scene.lights), 2.)
    lights = _abi.RmAreaLights()
    lights.n_lights, lights.radius, lights.samples = radii.shape[0], radii.ctypes.data_as(C.POINTER(C.c_double)), 2

    def call(samples=2, handle=hd, lt=lights, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        return L.rm_render_path(handle, C.byref(q), samples, None, None, C.byref(lt) if lt is not None else None, None, None,
                                out.ctypes.data, out8.ctypes.data, None)

    assert call() == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()
    assert call(handle=987654) == -3
    assert call(samples=9) == -3 and call(samples=0) == -3 and call(max_depth=0) == -3 and call(samples=3) == -3
    few = _abi.RmAreaLights()
    few.n_lights, few.radius, few.samples = radii.shape[0] - 1, radii.ctypes.data_as(C.POINTER(C.c_double)), 2
    assert call(lt=few) == -3                                   # n_lights differs from the scene's
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    q = _abi.RmParams.from_buffer_copy(p)
    q.width, q.height = 16384, 64
    assert L.rm_render_path(hd, C.byref(q), 8, None, None, None, None, None, wide.ctypes.data, None, None) == -4
    out[:] = 0
    out8[:] = 0
    assert call() == 0
    assert same(out, want) and np.array_equal(out8, want8)


def test_a_retained_delivery_after_a_path_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the path
    call in between wrote the frame too, so the library must forget that delivery."""
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
    r.render_path(fb, b, 2, light_radii=2., displacement=(0.5, 0., 0.))

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the demo frame lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)


def test_headless_harness_saves_the_path_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "path.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--path", "--depth", "4", "--light-radius", "2",
                        "--move", "1,0.5,0,0", "--aperture", "0.3", "--focus", "12", "--look-at", "1,0,-10", "--out", out],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    disp = np.zeros((len(scene.shapes), 3))
    disp[1] = (0.5, 0., 0.)
    rd = rm_gpu.create_renderer(1.5, h, w)
    rd.max_depth = 4
    rd.render_path(fb, scene, 3, forward=(1., 0., -10.), aperture=0.3, focus=12., light_radii=2., displacement=disp, rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--path", "--combine"], ["--path", "--indirect"], ["--path", "--contrast", "0.1"], ["--path", "--f64"],
                ["--path", "--rows-f64"], ["--indirect", "--combine"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
