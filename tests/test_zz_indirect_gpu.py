"""GPU part of the diffuse interreflection tests (see tests/test_indirect.py): rm_render_indirect against the oracle's indirect
frame (tests/indirect_ref.py) under the lens parity criterion, the routed cases and the never-hit anchor against rm_render_lens
(bit for bit), the furnace's closed form, the hierarchy, determinism, rows, the 8-bit frame, argument checks, retained-frame
bookkeeping and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import indirect_ref, lens_ref, view_ref
from tests import supersample_ref as SS
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def indirect(rm, scene, w, h, s, view=None, aperture=0., focus=1., accel=False, depth=3, rows=(0, -1), fill=0., cull=True):
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel, r.cull_backfacing = depth, accel, cull
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    fb.buffer[:] = fill
    b8 = np.zeros((h, w, 3), dtype=np.uint8)
    fwd, up = view if view is not None else (None, (0., 1., 0.))
    msg = r.render_indirect(fb, scene, s, forward=fwd, up=up, aperture=aperture, focus=focus, rgb8=b8, patch_rows=rows)
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


YAW30, PITCH = view_ref.VIEWS["yaw30"], view_ref.VIEWS["pitch-20"]
# (scene, width, height, max_depth, workload options, s, view, aperture, focus)
CASES = [("demo", 320, 256, 3, {}, 2, None, 0., 1.), ("demo", 320, 256, 3, {}, 4, None, 0., 1.),
         ("cornell_box", 320, 256, 3, {}, 2, None, 0., 1.), ("cornell_box", 320, 256, 4, {}, 3, YAW30, 0., 1.),
         ("ngons", 320, 192, 4, dict(n_spheres=12, n_polygons=40), 2, None, 0., 1.),
         ("stress", 320, 192, 4, dict(n_spheres=256, grid=24), 2, None, 0., 1.),
         ("demo", 320, 256, 3, {}, 3, YAW30, 0., 1.), ("demo", 320, 256, 3, {}, 3, PITCH, 0.4, 12.)]


@pytest.mark.parametrize("c", CASES, ids=["%s-s%d-%s%s" % (c[0], c[5], "view" if c[6] else "none", "-lens" if c[7] else "") for c in CASES])
def test_indirect_frames_meet_the_parity_criterion(rm_gpu, c):
    name, w, h, depth, kw, s, view, aperture, focus = c
    scene, oscene = scenes(name, **kw)
    basis = None if view is None else view_ref.numpy_basis(*view)
    ref = indirect_ref.render(oscene, w, h, s, basis=basis, aperture=aperture, focus=focus, max_depth=depth)
    accels = [False, True] if name in ("stress", "cornell_box") else [False]
    for accel in accels:
        got, got8, st = indirect(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth)
        r = lens_ref.check_parity(got, got8, ref, (h // 32) * 32)
        print(name, s, view is not None, accel, r)
        assert r["fragile_frac"] < 0.2, r
        assert st.kernel_launches == 2 and st.ms_total >= st.ms_render > 0
        assert not same(got, lens(rm_gpu, scene, w, h, s, view=view, aperture=aperture, focus=focus, accel=accel, depth=depth)[0])


@pytest.mark.parametrize("kind", ["depth1", "no-bounce"])
@pytest.mark.parametrize("view", [None, YAW30], ids=["none", "yaw30"])
def test_routed_calls_are_the_lens_frame(rm_gpu, kind, view):
    if kind == "depth1":
        scene, depth = scenes("stress", n_spheres=256, grid=24)[0], 1
    else:
        scene, depth = workloads.build_scene(indirect_ref.anchor_desc(with_target=False)), 5
    (got, got8, st), names = kernels_run(lambda: indirect(rm_gpu, scene, 320, 192, 3, view=view, aperture=0.5, focus=30.,
                                                           depth=depth))
    assert ran(names, "lens_kernel") and not ran(names, "indirect_kernel"), names      # routed to rm_render_lens
    want, want8, st0 = lens(rm_gpu, scene, 320, 192, 3, view=view, aperture=0.5, focus=30., depth=depth)
    assert same(got, want) and np.array_equal(got8, want8) and st.max_value == st0.max_value and got.any()


@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("cull", [False, True])
@pytest.mark.parametrize("spheres", [True, False], ids=["spheres", "planes"])
def test_the_kernel_is_the_lens_kernel_where_nothing_bounces(rm_gpu, accel, cull, spheres):
    scene = workloads.build_scene(indirect_ref.anchor_desc(spheres=spheres))
    for s, aperture in ((1, 0.), (3, 0.3)):
        (got, got8, st), names = kernels_run(lambda: indirect(rm_gpu, scene, 320, 192, s, aperture=aperture, focus=20., accel=accel,
                                                               depth=4, cull=cull))
        assert ran(names, "indirect_kernel") and not ran(names, "lens_kernel"), names      # not routed
        want, want8, _ = lens(rm_gpu, scene, 320, 192, s, aperture=aperture, focus=20., accel=accel, depth=4, cull=cull)
        assert same(got, want) and np.array_equal(got8, want8) and got.any()


@pytest.mark.parametrize("depth", [2, 3, 5])
def test_furnace_closed_form(rm_gpu, depth):
    rho = 0.6
    scene = workloads.build_scene(indirect_ref.furnace_desc(rho))
    (got, _, st), names = kernels_run(lambda: indirect(rm_gpu, scene, 256, 192, 3, depth=depth))
    assert ran(names, "indirect_kernel"), names
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
        scenes(name, **(dict(n_spheres=256, grid=24) if name == "stress" else {}))[0]
    a, a8, sa = indirect(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5)
    b, b8, sb = indirect(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5, accel=True)
    c, c8, _ = indirect(rm_gpu, scene, 320, 192, 3, view=YAW30, depth=5, accel=True)
    assert same(a, b) and np.array_equal(a8, b8) and sa.max_value == sb.max_value and a.any()
    assert same(b, c) and np.array_equal(b8, c8)


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene, _ = scenes("cornell_box")
    full, full8, _ = indirect(rm_gpu, scene, 320, 240, 3, fill=np.nan)
    assert np.isnan(full[224:]).all() and np.isfinite(full[:224]).all()
    part, part8, _ = indirect(rm_gpu, scene, 320, 240, 3, rows=(1, 4), fill=np.nan)
    assert np.isnan(part[:32]).all() and np.isnan(part[128:]).all() and not part8[:32].any() and not part8[128:].any()
    assert same(part[32:128], full[32:128]) and part8[32:128].any()


@pytest.mark.parametrize("view", [None, YAW30])
def test_rgb8_is_the_tone_map_of_the_float_rows(rm_gpu, view):
    scene, _ = scenes("demo")
    got, got8, st = indirect(rm_gpu, scene, 320, 240, 2, view=view)
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

    def call(samples=2, handle=hd, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, v in fields.items():
            setattr(q, k, v)
        return L.rm_render_indirect(handle, C.byref(q), None, None, samples, out.ctypes.data, out8.ctypes.data, None)

    assert call() == 0
    want, want8 = out.copy(), out8.copy()
    assert want.any()
    assert call(handle=987654) == -3
    assert call(samples=9) == -3 and call(samples=0) == -3 and call(max_depth=0) == -3
    wide = np.zeros((64, 16384, 3), dtype=np.float32)
    q = _abi.RmParams.from_buffer_copy(p)
    q.width, q.height = 16384, 64
    assert L.rm_render_indirect(hd, C.byref(q), None, None, 8, wide.ctypes.data, None, None) == -4
    out[:] = 0
    out8[:] = 0
    assert call() == 0
    assert same(out, want) and np.array_equal(out8, want8)


def test_a_retained_delivery_after_an_indirect_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    indirect call in between wrote the frame too, so the library must forget that delivery."""
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
    r.render_indirect(fb, b, 2)

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the demo frame lights tiles that are black in A's
    r.render(fb, a)
    assert same(fb.buffer, fresh_a)


def test_headless_harness_saves_the_indirect_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "indirect.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--samples", "3", "--indirect", "--aperture", "0.3",
                        "--focus", "12", "--look-at", "1,0,-10", "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    rm_gpu.create_renderer(1.5, h, w).render_indirect(fb, scene, 3, forward=(1., 0., -10.), aperture=0.3, focus=12., rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    for bad in (["--indirect", "--light-radius", "1"], ["--indirect", "--roughness", "0.2"], ["--indirect", "--move", "0,1,0,0"],
                ["--indirect", "--combine"], ["--indirect", "--contrast", "0.1"], ["--indirect", "--f64"], ["--indirect", "--rows-f64"]):
        assert subprocess.run([exe] + bad, capture_output=True).returncode == 2, bad
