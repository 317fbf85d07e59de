"""Path-traced frames (rm_render_path, include/rm_b200.h) without a GPU: the oracle's path-traced frame (tests/path_oracle.cpp)
against the two restatements it combines (tests/indirect_oracle.cpp, tests/distributed_oracle.cpp) and against a closed form,
and the path kernel's per-ray code compiled for the host (tests/emu/rm_path_emu.cpp) against the oracle and against the
indirect and distributed kernels' code.  GPU part: tests/test_zz_path_gpu.py."""
import ctypes as C
import math

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import distributed_ref, indirect_ref, lens_ref, path_ref, rough_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import distributed_emu, indirect_emu, lens_emu, path_emu
from tests.oracle_scenes import build_oracle_scene
from tests.test_distributed import area_radii, moving

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


def effects(scene, which, g=0.1, r=3.):
    e = {}
    if "area" in which:
        e["radii"] = area_radii(scene, r)
    if "rough" in which:
        e["roughness"] = np.where(rough_ref.glass_like(scene), g, 0.)
    if "motion" in which:
        e["disp"] = moving(scene)
    return e


# ---- the oracle's path-traced frame against the two restatements it combines ----
def test_oracle_frame_without_active_effects_is_the_indirect_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    w, h, depth = 96, 64, 4
    b = _basis(view_ref.VIEWS["yaw30"])
    zero_r, zero_g = np.zeros(len(scene.lights)), np.zeros(scene.num_prims)
    for s in (2, 3):
        want = indirect_ref.render(oscene, w, h, s, basis=b, aperture=0.3, focus=9., max_depth=depth)["rgb"]
        got = path_ref.render(oscene, w, h, s, radii=zero_r, roughness=zero_g, basis=b, aperture=0.3, focus=9., max_depth=depth)["rgb"]
        assert np.array_equal(got, want), s
    # s = 1: area_offset, rough_offset and motion_time are the identity, so every effect is inert
    one = indirect_ref.render(oscene, w, h, 1, basis=b, max_depth=depth)["rgb"]
    every = path_ref.render(oscene, w, h, 1, basis=b, max_depth=depth, **effects(scene, "area+rough+motion"))["rgb"]
    assert np.array_equal(every, one)


def test_oracle_frame_without_bounces_is_the_distributed_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    w, h, s = 96, 64, 3
    b = _basis(view_ref.VIEWS["yaw30"])
    e = effects(scene, "area+rough+motion")
    want = distributed_ref.render(oscene, w, h, s, basis=b, max_depth=1, **e)["rgb"]
    assert np.array_equal(path_ref.render(oscene, w, h, s, basis=b, max_depth=1, **e)["rgb"], want)
    assert not np.array_equal(path_ref.render(oscene, w, h, s, basis=b, max_depth=4, **e)["rgb"],
                              distributed_ref.render(oscene, w, h, s, basis=b, max_depth=4, **e)["rgb"])
    black = indirect_ref.anchor_desc(with_target=False)        # no primitive meets the bounce condition
    bscene, ob = workloads.build_scene(black), build_oracle_scene(black)
    e = effects(bscene, "area+rough+motion", g=0.2, r=2.)
    want = distributed_ref.render(ob, 128, 96, s, basis=b, aperture=0.3, focus=20., max_depth=4, **e)["rgb"]
    got = path_ref.render(ob, 128, 96, s, basis=b, aperture=0.3, focus=20., max_depth=4, **e)["rgb"]
    assert np.array_equal(got, want) and got.any()


# ---- the furnace: the camera inside a moving diffuse sphere, lit by nothing but the background ----
@pytest.mark.parametrize("depth", [2, 3, 4, 5])
def test_furnace_closed_form_with_every_effect_active(depth):
    rho = 0.6
    desc = indirect_ref.furnace_desc(rho)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    e = dict(radii=[5.], disp=[[3., -2., 1.5]])                # a black area light; the sphere moves, the camera stays inside
    want = indirect_ref.furnace_value(rho, depth)
    ref = path_ref.render(oscene, 64, 64, 3, max_depth=depth, **e)["rgb"]
    assert np.abs(ref / want - 1.).max() <= 1e-12
    for accel in (False, True):
        got = path_emu.render(scene, 64, 64, 3, max_depth=depth, accel=accel, **e)["rgb"].astype(np.float64)
        assert np.abs(got / want - 1.).max() <= 1e-6, accel


# ---- the path kernel's per-ray code, compiled for the host, against the oracle's path-traced frame ----
# (scene, width, height, max_depth, workload options, roughness of the glass-like primitives)
CASES = [("demo", 128, 96, 3, {}, 0.1), ("stress", 128, 96, 4, dict(n_spheres=64, grid=7), 0.05),
         ("ngons", 128, 96, 4, dict(n_spheres=12, n_polygons=40), 0.2), ("cornell_box", 128, 96, 3, {}, 0.1)]
# (effects, view, aperture, focus): each effect with the bounce under the pinhole, and all four with a turned view and a lens
COMBOS = {"area": ("area", None, 0., 1.), "rough": ("rough", None, 0., 1.), "motion": ("motion", None, 0., 1.),
          "all+yaw30+lens": ("area+rough+motion", view_ref.VIEWS["yaw30"], 0.3, 12.)}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw, g = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, workloads.build_scene(desc), build_oracle_scene(desc), g


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("combo", list(COMBOS))
def test_fp32_path_meets_the_parity_criterion(case, combo, s):
    name, w, h, depth, scene, oscene, g = case
    which, view, aperture, focus = COMBOS[combo]
    b = _basis(view)
    e = effects(scene, which, g)
    ref = path_ref.render(oscene, w, h, s, basis=b, aperture=aperture, focus=focus, max_depth=depth, **e)
    got = path_emu.render(scene, w, h, s, basis=b, aperture=aperture, focus=focus, max_depth=depth, cull=False, **e)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    dist = distributed_emu.render(scene, w, h, s, basis=b, aperture=aperture, focus=focus, max_depth=depth, cull=False, **e)["rgb"]
    assert not np.array_equal(got, dist)                        # the bounce adds light


# ---- the hierarchy (the swept one with motion) changes no pixel ----
BIT_CASES = [("demo", {}), ("cornell_box", {}), ("stress", dict(n_spheres=64, grid=7)), ("ngons", dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_hierarchy_changes_no_pixel(name, kw):
    scene = workloads.scene(name, **kw)
    b = _basis(view_ref.VIEWS["yaw30"])
    for which in ("area+motion", "area+rough+motion"):
        e = effects(scene, which, r=2.)
        a = path_emu.render(scene, 128, 96, 3, basis=b, max_depth=4, **e)["rgb"]
        c = path_emu.render(scene, 128, 96, 3, basis=b, max_depth=4, accel=True, **e)["rgb"]
        assert np.array_equal(a, c) and a.any(), which


# ---- the inert-effect anchor: rough glass that is active but never hit leaves the indirect frame ----
@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_inert_rough_triangle_leaves_the_indirect_frame(name, kw):
    scene, g = path_ref.with_inert_triangle(workloads.scene(name, **kw))
    b = _basis(view_ref.VIEWS["yaw30"])
    for cull in (False, True):
        for accel in (False, True):
            want = indirect_emu.render(scene, 128, 96, 3, basis=b, aperture=0.3, focus=12., max_depth=4, cull=cull, accel=accel)
            got = path_emu.render(scene, 128, 96, 3, roughness=g, basis=b, aperture=0.3, focus=12., max_depth=4, cull=cull, accel=accel)
            assert got["glass_mode"] == want["glass_mode"]
            assert got["rgb"].tobytes() == want["rgb"].tobytes() and got["rgb"].any(), (cull, accel)


# ---- the never-hit anchor: black opaque surfaces and one diffuse triangle no ray can reach ----
def anchor(spheres):
    scene = workloads.build_scene(indirect_ref.anchor_desc(spheres=spheres))
    v = np.zeros((scene.num_prims, 3))
    if spheres:
        v[0], v[1] = (0.5, -0.25, 0.75), (-0.75, 0.5, 0.25)      # the two spheres move; the walls and the target stay
    e = dict(radii=area_radii(scene, 2.), roughness=np.where(rough_ref.glass_like(scene), 0.2, 0.), disp=v)
    return scene, e


@pytest.mark.parametrize("spheres", [True, False], ids=["spheres", "planes"])
def test_never_hit_diffuse_triangle_leaves_the_distributed_frame(spheres):
    scene, e = anchor(spheres)
    for accel in (False, True):
        want = distributed_emu.render(scene, 128, 96, 3, aperture=0.3, focus=20., max_depth=4, cull=False, accel=accel, **e)
        got = path_emu.render(scene, 128, 96, 3, aperture=0.3, focus=20., max_depth=4, cull=False, accel=accel, **e)
        assert got["glass_mode"] == want["glass_mode"] and (spheres or got["glass_mode"] == 0)
        assert got["rgb"].tobytes() == want["rgb"].tobytes(), accel
    assert (want["rgb"] > 0.).any(axis=2).mean() > 0.3         # the black surfaces fill most of the frame


# ---- argument checks of the C ABI and of the Python mirror ----
_keep = []


def _struct(kind, n=4, value=0.5, samples=2, null=False):
    arr = np.full(max(3 * n, 3), value, dtype=np.float64)
    _keep.append(arr)
    ptr = None if null else arr.ctypes.data_as(C.POINTER(C.c_double))
    if kind == "lights":
        st = _abi.RmAreaLights()
        st.n_lights, st.radius, st.samples = n, ptr, samples
    elif kind == "rough":
        st = _abi.RmRoughGlass()
        st.n_prims, st.roughness, st.samples = n, ptr, samples
    else:
        st = _abi.RmMotion()
        st.n_prims, st.displacement, st.samples = n, ptr, samples
    return st


def _call(samples=2, params=None, view=None, lens=None, lights=None, rough=None, motion=None, rgb=True, rgb8=False):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    ref = lambda x: C.byref(x) if x is not None else None     # noqa: E731
    return L.rm_render_path(1, C.byref(p), samples, ref(view), ref(lens), ref(lights), ref(rough), ref(motion),
                            out.ctypes.data if rgb else None, out8.ctypes.data if rgb8 else None, None)


@pytest.mark.parametrize("kind", ["lights", "rough", "motion"])
@pytest.mark.parametrize("kw", [dict(n=-1), dict(null=True), dict(value=np.nan), dict(value=np.inf), dict(value=-1.), dict(samples=0),
                                dict(samples=9), dict(samples=3)])
def test_invalid_effect_structs_are_rejected(kind, kw):
    if kind == "motion" and kw.get("value") == -1.:
        kw = dict(value=-np.inf)                               # a negative displacement is valid
    assert _call(**{kind: _struct(kind, **kw)}) == INVALID


def test_invalid_samples_views_lenses_and_parameters_are_rejected():
    L = _abi.load()
    for s in (0, 9, -1):
        assert _call(samples=s) == INVALID, s
    bad = _abi.RmView()
    bad.forward[:] = [0., 1., 0.]
    bad.up[:] = [0., 2., 0.]
    assert _call(view=bad) == INVALID
    for ln in ((-0.1, 10., 2), (0.5, 0., 2), (np.nan, 10., 2), (0.5, 10., 3)):     # the last: lens->samples != samples
        assert _call(lens=lens_emu.lens(*ln)) == INVALID, ln
    assert _call(rgb=False) == INVALID
    for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
        setattr(p, field, value)
        assert _call(params=p) == INVALID, field
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 48, 64)
    assert _call(params=p) == DIMENSIONS
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 9024, 64)                  # the 8 x frame is wider than 65535
    assert _call(samples=8, params=p) == DIMENSIONS


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    assert _call() == NOT_INITIALISED
    assert _call(lights=_struct("lights", n=2), rough=_struct("rough"), motion=_struct("motion"), lens=lens_emu.lens(0.5, 10., 2)) == \
        NOT_INITIALISED


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(samples=True), dict(light_radii=-1.),
                                dict(light_radii=(1., 2., 3.)), dict(roughness=np.nan), dict(roughness=[0.1, 0.2]),
                                dict(displacement=[np.nan, 0., 0.]), dict(displacement=[0.1, 0.2]), dict(aperture=-1.), dict(focus=0.),
                                dict(aperture=math.nan), dict(forward=(0., 1., 0.), up=(0., 1., 0.)), dict(patch_rows=(0, -1, 2))])
def test_renderer_rejects_invalid_path_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(light_radii=1., roughness=0.1, displacement=(0.5, 0., 0.))
    args.update(kw)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_path(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **args)
