"""Distributed ray tracing (rm_render_distributed, include/rm_b200.h) without a GPU: rule 4's light stratum of the shared
definition code (rm::area_offset) against numpy and the oracle's restatement bit for bit, the oracle's distributed frame against
its single-effect frames, and the distributed kernel's per-ray code compiled for the host (tests/emu/rm_distributed_emu.cpp)
against the oracle and against the lens, rough-glass and motion kernels' code.  GPU part: tests/test_zz_distributed_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import distributed_ref, lens_ref, motion_ref, rough_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import distributed_emu, lens_emu, motion_emu, rough_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


# ---- rule 4's stratum: ((i + 2j + L) mod s, (i + 3j) mod s) on the unit disc ----
@pytest.mark.parametrize("s", range(1, 9))
def test_area_offset_is_the_definition_and_a_bijection(s):
    for level in range(1, 9):
        points = set()
        for i in range(s):
            for j in range(s):
                got = distributed_emu.area_offset(s, i, j, level)
                want = distributed_ref.numpy_area_offset(s, i, j, level)
                orc = distributed_ref.oracle_area_offset(s, i, j, level)
                assert np.array(got).tobytes() == np.array(want, dtype=np.float64).tobytes() == np.array(orc).tobytes(), (s, i, j, level)
                assert got[0] ** 2 + got[1] ** 2 <= 1. + 1e-15
                points.add(got)
        assert len(points) == s * s, (s, level)              # a bijection over the s^2 samples
    if s == 1:
        assert distributed_emu.area_offset(1, 0, 0, 1) == (0., 0.)


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


def moving(scene, scale=1., seed=7):
    """One displacement per shape, seeded, in multiples of 1/64 (exact in FP32), up to `scale` per component."""
    rng = np.random.default_rng(seed)
    v = np.round(rng.uniform(-scale, scale, size=(len(scene.shapes), 3)) * 64.) / 64.
    return motion_ref.per_prim(scene, v)


def area_radii(scene, r=3.):
    """Every light a point but the last, which is a sphere of radius r."""
    n = len(scene.lights)
    return np.array([0.] * (n - 1) + [r])


# ---- the oracle's distributed frame where a single effect is given ----
def test_oracle_distributed_frame_with_one_effect_is_that_effects_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    w, h, s, depth = 96, 64, 2, 4
    zero = np.zeros(len(scene.lights))
    g = np.where(rough_ref.glass_like(scene), 0.05, 0.)
    v = moving(scene)
    b = _basis(view_ref.VIEWS["yaw30"])
    lens = lens_ref.render(oscene, w, h, 0.3, 9., s, basis=b, max_depth=depth)["rgb"]
    assert np.array_equal(distributed_ref.render(oscene, w, h, s, radii=zero, basis=b, aperture=0.3, focus=9., max_depth=depth)["rgb"], lens)
    rough = rough_ref.render(oscene, w, h, g, s, basis=b, max_depth=depth)["rgb"]
    assert np.array_equal(distributed_ref.render(oscene, w, h, s, radii=zero, roughness=g, basis=b, max_depth=depth)["rgb"], rough)
    motion = motion_ref.render(oscene, w, h, v, s, basis=b, max_depth=depth)["rgb"]
    assert np.array_equal(distributed_ref.render(oscene, w, h, s, radii=zero, disp=v, basis=b, max_depth=depth)["rgb"], motion)
    one = lens_ref.render(oscene, w, h, 0., 1., 1, max_depth=depth)["rgb"]
    every = distributed_ref.render(oscene, w, h, 1, radii=area_radii(scene), roughness=g, disp=v, max_depth=depth)["rgb"]
    assert np.array_equal(every, one)
    assert not np.array_equal(distributed_ref.render(oscene, w, h, s, radii=area_radii(scene), max_depth=depth)["rgb"],
                              lens_ref.render(oscene, w, h, 0., 1., s, max_depth=depth)["rgb"])


# ---- the distributed kernel's per-ray code, compiled for the host, against the oracle's distributed frame ----
# (scene, width, height, max_depth, workload options, roughness of the glass-like primitives)
CASES = [("demo", 128, 96, 3, {}, 0.1), ("stress", 128, 96, 6, dict(n_spheres=64, grid=7), 0.05),
         ("ngons", 128, 96, 4, dict(n_spheres=12, n_polygons=40), 0.2)]
EFFECTS = ["area", "area+rough", "area+motion", "rough+motion", "area+rough+motion"]
CAMERAS = {"pinhole": (None, 0., 1.), "yaw30+lens": (view_ref.VIEWS["yaw30"], 0.3, 12.)}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw, g = request.param
    desc = workloads.describe(name, **kw)
    scene = workloads.build_scene(desc)
    return name, w, h, depth, scene, build_oracle_scene(desc), g


def effects(scene, which, g=0.1, r=3.):
    e = {}
    if "area" in which:
        e["radii"] = area_radii(scene, r)
    if "rough" in which:
        e["roughness"] = np.where(rough_ref.glass_like(scene), g, 0.)
    if "motion" in which:
        e["disp"] = moving(scene)
    return e


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("which", EFFECTS)
@pytest.mark.parametrize("camera", list(CAMERAS))
def test_fp32_distributed_path_meets_the_parity_criterion(case, which, camera, s):
    name, w, h, depth, scene, oscene, g = case
    view, aperture, focus = CAMERAS[camera]
    b = _basis(view)
    e = effects(scene, which, g)
    ref = distributed_ref.render(oscene, w, h, s, basis=b, aperture=aperture, focus=focus, max_depth=depth, **e)
    got = distributed_emu.render(scene, w, h, s, basis=b, aperture=aperture, focus=focus, max_depth=depth, cull=False, **e)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    lens = lens_emu.render(scene, w, h, aperture, focus, s, basis=b, max_depth=depth, cull=False)["rgb"]
    assert not np.array_equal(got, lens)


# ---- with every radius 0 the distributed code is the lens, rough-glass and motion code bit for bit ----
BIT_CASES = [("demo", {}), ("cornell_box", {}), ("stress", dict(n_spheres=64, grid=7)), ("ngons", dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_zero_radii_are_the_single_effect_code_bit_for_bit(name, kw):
    scene = workloads.scene(name, **kw)
    w, h, s, depth = 128, 96, 3, 4
    b = _basis(view_ref.VIEWS["yaw30"])
    zero = np.zeros(len(scene.lights))
    g = np.where(rough_ref.glass_like(scene), 0.1, 0.)
    v = moving(scene)
    for accel in (False, True):
        kw2 = dict(basis=b, max_depth=depth, accel=accel)
        got = distributed_emu.render(scene, w, h, s, radii=zero, aperture=0.3, focus=12., **kw2)["rgb"]
        want = lens_emu.render(scene, w, h, 0.3, 12., s, **kw2)["rgb"]
        assert got.tobytes() == want.tobytes() and got.any(), ("lens", accel)
        if g.any():
            got = distributed_emu.render(scene, w, h, s, radii=zero, roughness=g, **kw2)["rgb"]
            want = rough_emu.render(scene, w, h, g, s, **kw2)["rgb"]
            assert got.tobytes() == want.tobytes(), ("rough", accel)
        got = distributed_emu.render(scene, w, h, s, radii=zero, disp=v, **kw2)["rgb"]
        want = motion_emu.render(scene, w, h, v, s, **kw2)["rgb"]
        assert got.tobytes() == want.tobytes(), ("motion", accel)


# ---- the hierarchy (the scene's, or the swept one with motion) changes no pixel ----
@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_hierarchy_changes_no_pixel(name, kw):
    scene = workloads.scene(name, **kw)
    b = _basis(view_ref.VIEWS["yaw30"])
    for which in ("area", "area+rough+motion"):
        e = effects(scene, which, r=2.)
        a = distributed_emu.render(scene, 128, 96, 3, basis=b, max_depth=4, **e)["rgb"]
        c = distributed_emu.render(scene, 128, 96, 3, basis=b, max_depth=4, accel=True, **e)["rgb"]
        assert np.array_equal(a, c), which


def test_a_scene_of_nine_lights_stays_on_brute_force():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    desc["lights"] = list(desc["lights"]) + [((10. * k - 40., 30., 10.), (1., 0.8, 0.6), 0.3) for k in range(9 - len(desc["lights"]))]
    scene = workloads.build_scene(desc)
    assert len(scene.lights) == 9
    e = dict(radii=np.full(9, 0.5), disp=moving(scene))
    a = distributed_emu.render(scene, 128, 96, 2, max_depth=3, **e)["rgb"]
    c = distributed_emu.render(scene, 128, 96, 2, max_depth=3, accel=True, **e)["rgb"]
    assert np.array_equal(a, c) and a.any()


# ---- a soft shadow of a moving occluder: the penumbra widens with the radius ----
MATTE = dict(diffusion=1., diffuse_color=(0.8, 0.8, 0.8), specular=0., specular_exponent=30., is_glass_like=False, reflection=0.95,
             refractive_index=1.)


def _shadow_scene(occluder=True):
    """A diffuse wall facing the camera, one light in front of it and a sphere between them that moves sideways."""
    quad = [(-12., -9., -20.), (12., -9., -20.), (12., 9., -20.), (-12., 9., -20.)]          # CCW in XY: normal +z
    spheres = [((3., -1.5, -13.), 1.5, MATTE)] if occluder else []
    desc = {"name": "shadow", "default": False, "spheres": spheres, "polygons": [(quad, MATTE)], "meshes": [],
            "lights": [((6., -3., -6.), (1., 1., 1.), 1.)]}
    scene = workloads.build_scene(desc)
    return scene, motion_ref.per_prim(scene, [[0.75, 0., 0.]] * len(scene.shapes)) if occluder else np.zeros((1, 3))


def test_penumbra_of_a_moving_occluder_grows_with_the_radius_and_a_tiny_light_is_the_point_light():
    (scene, v), (bare, v0) = _shadow_scene(), _shadow_scene(occluder=False)
    w, h, s = 160, 128, 4
    point = distributed_emu.render(scene, w, h, s, radii=[0.], disp=v, cull=False)["rgb"]
    lit = distributed_emu.render(bare, w, h, s, radii=[0.], disp=v0, cull=False)["rgb"].max(axis=2)
    wall = lit > 0.1 + 1e-4
    assert wall.sum() > 2000 and (wall & (point.max(axis=2) <= 0.1 + 1e-6)).sum() > 100     # a shadow the mover leaves dark
    counts = []
    for radius in (0.3, 1., 2.5):
        f = distributed_emu.render(scene, w, h, s, radii=[radius], disp=v, cull=False)["rgb"].max(axis=2)
        bare_f = distributed_emu.render(bare, w, h, s, radii=[radius], disp=v0, cull=False)["rgb"].max(axis=2)
        partial = wall & (f > 0.1 + 1e-4) & (f < bare_f * (1. - 1e-4))      # strictly between fully shadowed and fully lit
        counts.append(int(partial.sum()))
    assert counts[0] < counts[1] < counts[2], counts
    tiny = distributed_emu.render(scene, w, h, s, radii=[1e-6], disp=v, cull=False)["rgb"]
    assert np.abs(tiny.astype(np.float64) - point).max() <= 1e-4


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
    return L.rm_render_distributed(1, C.byref(p), samples, ref(view), ref(lens), ref(lights), ref(rough), ref(motion),
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
                                dict(forward=(0., 1., 0.), up=(0., 1., 0.)), dict(patch_rows=(0, -1, 2))])
def test_renderer_rejects_invalid_distributed_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(light_radii=1., roughness=0.1, displacement=(0.5, 0., 0.))
    args.update(kw)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_distributed(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **args)
