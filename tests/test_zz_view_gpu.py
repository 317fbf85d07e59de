"""GPU part of the camera-orientation tests (see tests/test_view.py): rm_render_view against rm_render for the identity view,
against the oracle's turned camera (tests/view_ref.py) under the parity criteria for five views, the FP64 validation
kernels bit for bit, the hierarchy on against off, rows, the device variant, argument checks, retained-frame bookkeeping
and the headless harness."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import parity, view_ref
from tests.oracle_scenes import build_oracle_scene

pytestmark = pytest.mark.gpu
VIEWS = view_ref.VIEWS


def same(a, b):
    return a.dtype == b.dtype and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def render(rm, scene, w, h, view=None, accel=False, depth=3, f64=False, counters=False, rows=(0, -1), fill=0.):
    """rm_render (view None) or rm_render_view: float frame, ids, 8-bit frame, stats."""
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    if f64:
        r.precision = _abi.RM_FP64
    fb = rm.create_frame_buffer(w, h, dtype=np.float64 if f64 else np.float32)
    fb.buffer[:] = fill
    ids = np.full((h, w), -7, dtype=np.int32)
    b8 = np.full((h, w, 3), 7, dtype=np.uint8)
    if view is None:
        r.render(fb, scene, prim_id=ids, rgb8=b8, counters=counters, patch_rows=rows)
    else:
        if counters:                                            # (render_view has no counters switch: through the ABI)
            p = r.params(fb, scene, rows)
            st = _abi.RmStats()
            st.pixels = 1
            fn = _abi.load().rm_render_view_f64 if f64 else _abi.load().rm_render_view
            _abi.check(fn(scene.device_handle(), C.byref(p), C.byref(rm.renderer._view(*view)), fb.buffer.ctypes.data,
                          ids.ctypes.data, b8.ctypes.data, C.byref(st)))
            r.last_stats = st
        else:
            r.render_view(fb, scene, view[0], view[1], prim_id=ids, rgb8=b8, patch_rows=rows)
    return {"rgb": fb.buffer, "prim_id": ids, "rgb8": b8, "stats": r.last_stats}


def scene_of(name, **kw):
    return workloads.build_scene(workloads.describe(name, **kw))


TEST_SIZES = {"demo": (320, 256, {}), "cornell_box": (320, 256, {}), "dodecahedron": (320, 256, {}),
              "stress": (320, 192, dict(n_spheres=256, grid=24)), "ngons": (320, 192, {})}


@pytest.mark.parametrize("accel", [False, True])
@pytest.mark.parametrize("name", sorted(TEST_SIZES))
def test_identity_view_is_rm_render(rm_gpu, name, accel):
    w, h, kw = TEST_SIZES[name]
    scene = scene_of(name, **kw)
    a = render(rm_gpu, scene, w, h, accel=accel)
    for view in (view_ref.IDENTITY, ((0., 0., -3.), (0., 0.5, 0.))):
        b = render(rm_gpu, scene, w, h, view=view, accel=accel)
        assert same(a["rgb"], b["rgb"]) and np.array_equal(a["prim_id"], b["prim_id"]) and np.array_equal(a["rgb8"], b["rgb8"])


PARITY = [("demo", 1600, 1280, 3, {}), ("cornell_box", 1920, 1088, 3, {}), ("stress", 320, 192, 6, dict(n_spheres=256, grid=24)),
          ("ngons", 320, 192, 4, {})]


@pytest.fixture(scope="module", params=PARITY, ids=[c[0] for c in PARITY])
def case(request):
    name, w, h, depth, kw = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, workloads.build_scene(desc), build_oracle_scene(desc)


@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_views_meet_the_parity_criteria(rm_gpu, case, view):
    name, w, h, depth, scene, oscene = case
    ref = view_ref.render(oscene, w, h, view=VIEWS[view], max_depth=depth)
    got = render(rm_gpu, scene, w, h, view=VIEWS[view], depth=depth)
    print(name, view, parity.check_fp32(got, ref, (h // 32) * 32, got["rgb8"]))
    if name in ("stress", "ngons"):                            # the hierarchy under the view: the same frame, bit for bit
        b = render(rm_gpu, scene, w, h, view=VIEWS[view], depth=depth, accel=True)
        assert same(got["rgb"], b["rgb"]) and np.array_equal(got["prim_id"], b["prim_id"]) and np.array_equal(got["rgb8"], b["rgb8"])


F64 = [("demo", 256, 160, 3, {}), ("stress", 160, 128, 6, dict(n_spheres=64, grid=7)), ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
@pytest.mark.parametrize("name,w,h,depth,kw", F64, ids=[c[0] for c in F64])
def test_fp64_view_kernels_match_the_oracle(rm_gpu, name, w, h, depth, kw, view):
    desc = workloads.describe(name, **kw)
    ref = view_ref.render(build_oracle_scene(desc), w, h, view=VIEWS[view], max_depth=depth)
    got = render(rm_gpu, workloads.build_scene(desc), w, h, view=VIEWS[view], depth=depth, f64=True, counters=True)
    parity.check_exact(got, ref, rel=1e-13)
    st = got["stats"]
    # cull_backfacing is on: the same control flow, fewer plane tests (as test_fp64_kernels_match_the_oracle)
    for k in ("pixels", "closest_segments", "anyhit_segments", "hits", "light_evals", "lit_lights", "glass_hits",
              "reflections", "refractions", "sphere_tests", "sphere_hits"):
        assert getattr(st, k) == ref["counters"][k], k


def test_triangle_only_scene_with_tile_schedule(rm_gpu):
    """The dodecahedron (a few triangles: K0 classifies tiles on the rotated records and empty tiles are skipped)."""
    desc = workloads.describe("dodecahedron")
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    w, h = 640, 480
    for view in (VIEWS["yaw30"], VIEWS["roll90"], ((0.1, 0.05, -1.), (0.2, 1., 0.))):
        ref = view_ref.render(oscene, w, h, view=view)
        got = render(rm_gpu, scene, w, h, view=view)
        parity.check_fp32(got, ref, h, got["rgb8"])
        assert (got["prim_id"] >= 0).any()


def test_rows_equal_the_full_frame_and_the_rest_is_untouched(rm_gpu):
    scene = scene_of("demo")
    w, h = 320, 256
    v = VIEWS["yaw30"]
    full = render(rm_gpu, scene, w, h, view=v)
    part = render(rm_gpu, scene, w, h, view=v, rows=(2, 5), fill=0.5)
    assert same(part["rgb"][64:160], full["rgb"][64:160]) and np.array_equal(part["prim_id"][64:160], full["prim_id"][64:160])
    assert (part["rgb"][:64] == 0.5).all() and (part["rgb"][160:] == 0.5).all()
    assert (part["prim_id"][:64] == -7).all() and (part["prim_id"][160:] == -7).all() and (part["rgb8"][160:] == 7).all()


@pytest.mark.parametrize("accel", [False, True])
def test_device_variant_equals_the_host_variant(rm_gpu, accel):
    import torch
    scene = scene_of("stress", n_spheres=256, grid=24)
    w, h = 320, 192
    v = VIEWS["pitch-20"]
    host = render(rm_gpu, scene, w, h, view=v, accel=accel, depth=6)
    r = rm_gpu.create_renderer(1.5, h, w)
    r.max_depth, r.accel = 6, accel
    p = r.params(rm_gpu.create_frame_buffer(w, h), scene)
    d_rgb = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
    d_ids = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    d_max = torch.zeros(1, dtype=torch.float32, device="cuda")
    _abi.check(_abi.load().rm_render_view_device(scene.device_handle(), C.byref(p), C.byref(rm_gpu.renderer._view(*v)),
                                                 d_rgb.data_ptr(), d_ids.data_ptr(), d_max.data_ptr(), None))
    torch.cuda.synchronize()
    assert same(d_rgb.cpu().numpy(), host["rgb"]) and np.array_equal(d_ids.cpu().numpy(), host["prim_id"])
    assert float(d_max.item()) == host["stats"].max_value


def test_argument_checks(rm_gpu):
    rm = rm_gpu
    scene = scene_of("demo")
    L = _abi.load()
    w, h = 128, 96
    p = rm.create_renderer(1.5, h, w).params(rm.create_frame_buffer(w, h), scene)
    hd = scene.device_handle()
    out = np.zeros((h, w, 3), dtype=np.float32)
    out64 = np.zeros((h, w, 3), dtype=np.float64)
    v = rm.renderer._view(*VIEWS["yaw30"])

    def call(view=v, handle=hd, fn=L.rm_render_view, rgb=out, **fields):
        q = _abi.RmParams.from_buffer_copy(p)
        for k, val in fields.items():
            setattr(q, k, val)
        return fn(handle, C.byref(q), C.byref(view) if view is not None else None, rgb.ctypes.data, None, None, None)

    assert call() == 0 and out.any()
    assert call(view=None) == -3
    assert call(view=rm.renderer._view((0., 1., 0.), (0., 2., 0.))) == -3
    assert call(view=rm.renderer._view((0., 0., 0.), (0., 1., 0.))) == -3
    assert call(view=rm.renderer._view((np.nan, 0., -1.), (0., 1., 0.))) == -3
    assert call(precision=_abi.RM_FP64) == -3
    assert call(fn=L.rm_render_view_f64, rgb=out64) == -3                 # precision RM_FP32 in the params
    assert call(fn=L.rm_render_view_f64, rgb=out64, precision=_abi.RM_FP64) == 0
    assert call(handle=987654) == -3
    assert call(width=100) == -4
    assert call(max_depth=9) == -3
    assert L.rm_render_view_device(hd, C.byref(p), None, None, None, None, None) == -3
    fb = rm.create_frame_buffer(w, h)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, h, w).render_view(fb, scene, (0., 1., 0.), (0., 1., 0.))


def test_a_retained_delivery_after_a_view_frame_clears_what_it_left(rm_gpu):
    """rm_render_rows_f32(RM_ROWS_RETAINED) only clears the tiles its own previous delivery into the frame left busy; the
    view call in between wrote the frame too, so the library must forget that delivery."""
    rm = rm_gpu
    w, h = 640, 480
    a = scene_of("cornell_box")
    fresh_a = render(rm, a, w, h)["rgb"]
    r = rm.create_renderer(1.5, h, w)
    r.retained = True
    fb = rm.create_frame_buffer(w, h, dtype=np.float32)
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)
    r.render_view(fb, a, (0.35, -0.2, -1.), (0., 1., 0.))

    def lit_tiles(f):
        return (f[:480].reshape(15, 32, 20, 32, 3) != 0).any(axis=(1, 3, 4))
    assert (lit_tiles(fb.buffer) & ~lit_tiles(fresh_a)).sum() >= 10        # the turned camera lights tiles that are black in A's
    r.render(fb, a)
    assert np.array_equal(fb.buffer, fresh_a)


def test_headless_harness_saves_the_view_frame(rm_gpu, tmp_path):
    from rusty_marcher_b200 import build as bld
    from rusty_marcher_b200.renderer import look_at
    exe = bld.build_examples()
    w, h = 320, 256
    out = str(tmp_path / "view.ppm")
    r = subprocess.run([exe, "--width", str(w), "--height", str(h), "--camera", "0", "0", "-20", "--look-at", "6,-0.5,-18",
                        "--up", "0,1,0.2", "--accel", "--out", out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    scene = rm_gpu.Scene.create_default()
    scene.offset_camera((0., 0., -20.))
    fb = rm_gpu.create_frame_buffer(w, h)
    rgb8 = np.zeros((h, w, 3), dtype=np.uint8)
    ren = rm_gpu.create_renderer(1.5, h, w)
    ren.accel = True
    ren.render_view(fb, scene, look_at((0., 0., -20.), (6., -0.5, -18.)), (0., 1., 0.2), rgb8=rgb8)
    mine = str(tmp_path / "py.ppm")
    assert _abi.load().rm_write_ppm(os.fsencode(mine), w, h, rgb8.ctypes.data) == 0
    assert open(out, "rb").read() == open(mine, "rb").read()
    assert rgb8.any()
    assert subprocess.run([exe, "--look-at", "1,2,3", "--samples", "2"], capture_output=True).returncode == 2
    assert subprocess.run([exe, "--look-at", "1,2"], capture_output=True).returncode == 2
