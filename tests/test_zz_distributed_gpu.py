"""GPU part of the distributed ray tracing tests (see tests/test_distributed.py): rm_render_distributed against the oracle's
distributed frame (tests/distributed_ref.py) under the lens parity criterion, the routed cases against rm_render_lens,
rm_render_rough_glass and rm_render_motion (bit for bit), the kernel against those calls' kernels through a black area light,
the hierarchy against brute force, determinism, rows, the 8-bit frame, argument checks, retained-frame bookkeeping and the
headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from rusty_marcher_b200.lights import Light
from rusty_marcher_b200.obj import Obj
from tests import distributed_ref, lens_ref, motion_ref, rough_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _renderer(rm, w, h, depth, accel, cull):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel, r.cull_backfacing = depth, accel, cull
    return r


def _frame(rm, w, h, fill=0.):
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    return fb, np.zeros((h, w, 3), dtype=np.uint8)


def distributed(rm, scene, w, h, s, view=None, aperture=0., focus=1., radii=None, roughness=None, disp=None, accel=False, depth=3,
                rows=(0, -1), fill=0., cull=True):
    r = _renderer(rm, w, h, depth, accel, cull)
    fb, b8 = _frame(rm, w, h, fill)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_distributed(fb, scene, s, forward=fwd, up=up, aperture=aperture, focus=focus, light_radii=radii, roughness=roughness,
                               displacement=disp, rgb8=b8, patch_rows=rows)
    assert msg.startswith("Scene rendered in ")
    return fb.buffer, b8, r.last_stats


def single(rm, kind, scene, w, h, s, view=None, aperture=0., focus=1., roughness=None, disp=None, accel=False, depth=3, cull=True):
    """rm_render_lens, rm_render_rough_glass or rm_render_motion through the Renderer"""
    r = _renderer(rm, w, h, depth, accel, cull)
    fb, b8 = _frame(rm, w, h)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    if kind == "lens":
        r.render_lens(fb, scene, aperture, focus, s, forward=fwd, up=up, rgb8=b8)
    elif kind == "rough":
        r.render_rough_glass(fb, scene, roughness, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8)
    else:
        r.render_motion(fb, scene, disp, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8)
    return fb.buffer, b8, r.last_stats


def scenes(name, **kw):
    desc = workloads.describe(name, **kw)
    return workloads.build_scene(desc), build_oracle_scene(desc)


def per_shape(scene, scale=1., seed=7):
    """one seeded displacement per shape, in multiples of 1/64 (exact in FP32)"""
    rng = np.random.default_rng(seed)
    return np.round(rng.uniform(-scale, scale, size=(len(scene.shapes), 3)) * 64.) / 64.


def radii_of(scene, r=3.):
    return [0.] * (len(scene.lights) - 1) + [r]


def rough_of(scene, g):
    """g on every glass-like shape (an Obj counts as glass-like if any of its triangles is), 0 elsewhere, per shape"""
    out, k = [], 0
    gl = rough_ref.glass_like(scene)
    for sh in scene.shapes:
        n = sh.triangles.shape[0] if isinstance(sh, Obj) else 1
        out.append(g if gl[k:k + n].any() else 0.)
        k += n
    return np.array(out)


YAW30, PITCH = view_ref.VIEWS["yaw30"], view_ref.VIEWS["pitch-20"]
# (scene, width, height, max_depth, workload options, s, effects, view, aperture, focus, roughness)
CASES = [("demo", 320, 256, 3, {}, 2, "area", None, 0., 1., 0.1),
         ("demo", 320, 256, 3, {}, 4, "area+rough", None, 0., 1., 0.1),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 2, "area+motion", None, 0., 1., 0.2),
         ("stress", 320, 192, 6, dict(n_spheres=256, grid=24), 2, "rough+motion", None, 0., 1., 0.05),
         ("demo", 320, 256, 3, {}, 3, "area+rough+motion", YAW30, 0.4, 12., 0.1),
         ("stress", 320, 192, 6, dict(n_spheres=256, grid=24), 3, "area+rough+motion", PITCH, 0.3, 40., 0.05)]


@pytest.mark.parametrize("c", CASES, ids=["%s-s%d-%s%s" % (c[0], c[5], c[6], "-view-lens" if c[7] else "") for c in CASES])
def test_distributed_frames_meet_the_parity_criterion(rm_gpu, c):
    name, w, h, depth, kw, s, which, view, aperture, focus, g = c
    scene, oscene = scenes(name, **kw)
    e = {}
    if "area" in which:
        e["radii"] = radii_of(scene)
    if "rough" in which:
        e["roughness"] = rough_of(scene, g)
    if "motion" in which:
        e["disp"] = per_shape(scene)
    basis = None if view is None else view_ref.numpy_basis(*view)
    ref = distributed_ref.render(oscene, w, h, s, radii=e.get("radii"), basis=basis, aperture=aperture, focus=focus, max_depth=depth,
                                 roughness=None if "roughness" not in e else motion_ref.per_prim(scene, e["roughness"][:, None])[:, 0],
                                 disp=None if "disp" not in e else motion_ref.per_prim(scene, e["disp"]))
    for accel in ([False, True] if name == "stress" else [False]):
        got, got8, st = distributed(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth, cull=False,
                                    **e)
        print(name, s, which, view is not None, accel, lens_ref.check_parity(got, got8, ref, (h // 32) * 32))
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        lens = single(rm_gpu, "lens", scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth, cull=False)[0]
        assert not same(got, lens)


@pytest.mark.parametrize("kind", ["s1", "none", "zero-radii", "rough", "motion"])
@pytest.mark.parametrize("view", [None, YAW30], ids=["none", "yaw30"])
def test_routed_calls_are_the_single_effect_frames(rm_gpu, kind, view):
    scene, _ = scenes("demo")
    w, h, depth = 320, 192, 5
    g, v = rough_of(scene, 0.1), per_shape(scene)
    s = 1 if kind == "s1" else 3
    lens_kw = dict(view=view, aperture=0.5, focus=12., depth=depth)
    if kind == "s1":
        got = distributed(rm_gpu, scene, w, h, s, radii=radii_of(scene), roughness=g, disp=v, **lens_kw)
        want = single(rm_gpu, "lens", scene, w, h, s, **lens_kw)
    elif kind == "none":
        got = distributed(rm_gpu, scene, w, h, s, **lens_kw)
        want = single(rm_gpu, "lens", scene, w, h, s, **lens_kw)
    elif kind == "zero-radii":
        got = distributed(rm_gpu, scene, w, h, s, radii=[0.] * len(scene.lights), roughness=np.zeros(len(scene.shapes)),
                          disp=np.zeros((len(scene.shapes), 3)), **lens_kw)
        want = single(rm_gpu, "lens", scene, w, h, s, **lens_kw)
    elif kind == "rough":
        got = distributed(rm_gpu, scene, w, h, s, radii=[0.] * len(scene.lights), roughness=g, **lens_kw)
        want = single(rm_gpu, "rough", scene, w, h, s, roughness=g, **lens_kw)
    else:
        got = distributed(rm_gpu, scene, w, h, s, roughness=np.zeros(len(scene.shapes)), disp=v, **lens_kw)
        want = single(rm_gpu, "motion", scene, w, h, s, disp=v, **lens_kw)
    assert same(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2].max_value == want[2].max_value and got[0].any()


def with_black_light(name, **kw):
    """The scene plus one light of colour (0, 0, 0) (built without create_light's normalisation): as an area light it forces the
    distributed kernel and adds exactly +0 to every sum."""
    scene, _ = scenes(name, **kw)
    scene.lights.append(Light((4., 6., -2.), (0., 0., 0.), 1.0))
    return scene


@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("cull", [True, False])
def test_the_kernel_is_the_single_effect_kernels_through_a_black_area_light(rm_gpu, accel, cull):
    scene = with_black_light("demo")
    w, h, s, depth = 320, 192, 3, 5
    black = [0.] * (len(scene.lights) - 1) + [2.]
    g, v = rough_of(scene, 0.1), per_shape(scene)
    kw = dict(view=YAW30, depth=depth, accel=accel, cull=cull)
    for kind, e in (("rough", dict(roughness=g)), ("motion", dict(disp=v)), ("lens", dict(aperture=0.3, focus=12.))):
        got, got8, st = distributed(rm_gpu, scene, w, h, s, radii=black, **e, **kw)
        assert st.kernel_launches == 2                             # the distributed kernel ran (no routing)
        want, want8, st0 = single(rm_gpu, kind, scene, w, h, s, **e, **kw)
        assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value and got.any(), kind


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
    e = dict(radii=[1.] * len(scene.lights), roughness=rough_of(scene, 0.1))
    for disp in (None, per_shape(scene, 2.)):
        a, a8, sa = distributed(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=6, disp=disp, **e)
        b, b8, sb = distributed(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=6, disp=disp, accel=True, **e)
        c, c8, _ = distributed(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=6, disp=disp, accel=True, **e)
        assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()
        assert same(b, c) and np.array_equal(b8, c8)


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("demo")
    e = dict(radii=radii_of(scene), roughness=rough_of(scene, 0.1), disp=per_shape(scene))
    full, full8, _ = distributed(rm_gpu, scene, 320, 240, 3, fill=np.nan, **e)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = distributed(rm_gpu, scene, 320, 240, 3, rows=(1, 4), fill=np.nan, **e)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, YAW30])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = distributed(rm_gpu, scene, 320, 240, 2, view=view, radii=radii_of(scene), disp=per_shape(scene))
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
    n, nl = scene.num_prims, len(scene.lights)
    out = np.zeros((h, w, 3), dtype=np.float32)
    out8 = np.zeros((h, w, 3), dtype=np.uint8)
    v = np.ascontiguousarray(np.tile([0.5, 0.25, -0.5], (n + 1, 1)))
    g = np.full(n + 1, 0.1)
    r = np.full(nl + 1, 1.)

    def call(n_lights=nl, n_rough=n, n_motion=n, samples=2, handle=hd, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, val in fields.items():
            setattr(q, k, val)
        al = _abi.RmAreaLights()
        al.n_lights, al.radius, al.samples = n_lights, r.ctypes.data_as(C.POINTER(C.c_double)), samples
        rg = _abi.RmRoughGlass()
        rg.n_prims, rg.roughness, rg.samples = n_rough, g.ctypes.data_as(C.POINTER(C.c_double)), samples
        m = _abi.RmMotion()
        m.n_prims, m.displacement, m.samples = n_motion, v.ctypes.data_as(C.POINTER(C.c_double)), samples
        return L.rm_render_distributed(handle, C.byref(q), samples, None, None, C.byref(al), C.byref(rg), C.byref(m), out.ctypes.data,
                                       out8.ctypes.data, None)

    assert call() == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()
    assert call(n_lights=nl + 1) == -3 and call(n_lights=nl - 1) == -3
    assert call(n_rough=n + 1) == -3 and call(n_motion=n - 1) == -3
    assert call(handle=987654) == -3
    assert call(samples=9) == -3 and call(max_depth=0) == -3
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    q = _abi.RmParams.from_buffer_copy(p)
    q.width, q.height = 16384, 64
    assert L.rm_render_distributed(hd, C.byref(q), 8, None, None, None, None, None, wide.ctypes.data, None, None) == -4
    out[:] = 0
    out8[:] = 0
    assert call() == 0
    assert same(out, want) and np.array_equal(out8, want8)


def test_a_retained_delivery_after_a_distributed_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    distributed call in between wrote the frame too, so the library must forget that delivery."""
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
    r.render_distributed(fb, b, 2, light_radii=1., displacement=(1., 0., 0.))

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the demo frame lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)


def test_headless_harness_saves_the_distributed_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "distributed.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--combine", "--move", "0,1.5,-0.5,0",
                        "--light-radius", "0,4", "--roughness", "0.1", "--aperture", "0.3", "--focus", "12", "--look-at", "1,0,-10",
                        "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    disp = np.zeros((len(scene.shapes), 3))
    disp[0] = (1.5, -0.5, 0.)
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_distributed(fb, scene, 3, forward=(1., 0., -10.), aperture=0.3, focus=12.,
                                                          light_radii=(0., 4.), roughness=0.1, displacement=disp, rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--combine", "--move", "0,1,0,0", "--contrast", "0.1"], ["--combine", "--light-radius", "1", "--f64"],
                ["--combine", "--roughness", "0.1", "--rows-f64"], ["--move", "0,1,0,0", "--roughness", "0.2"],
                ["--light-radius", "1", "--aperture", "0.3", "--focus", "12"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
