"""Motion blur (rm_render_motion, include/rm_b200.h RmMotion) without a GPU: the sample times of the shared definition code
(rm::motion_time) against numpy and the oracle's restatement bit for bit, the oracle's motion frame against its lens frame where
nothing moves, the swept hierarchy, and the motion kernel's per-ray code compiled for the host (tests/emu/rm_motion_emu.cpp)
against the oracle and against the lens kernel's.  GPU part: tests/test_zz_motion_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from rusty_marcher_b200.obj import Obj
from tests import lens_ref, motion_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import emu, lens_emu, motion_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


# ---- the sample times: m = s ((2i + j) mod s) + ((i + j) mod s), tau = (m + 0.5) / s^2 - 0.5 ----
@pytest.mark.parametrize("s", range(1, 9))
def test_motion_time_is_the_definition_and_a_bijection(s):
    taus = []
    for i in range(s):
        for j in range(s):
            got = motion_emu.motion_time(s, i, j)
            want = motion_ref.numpy_motion_time(s, i, j)
            assert np.float64(got).tobytes() == want.tobytes() == np.float64(motion_ref.oracle_motion_time(s, i, j)).tobytes(), (s, i, j)
            assert -0.5 < got < 0.5
            taus.append(got)
    strata = sorted(int(round((t + 0.5) * s * s - 0.5)) for t in taus)
    assert strata == list(range(s * s))                        # a bijection onto [0, s^2)
    assert abs(sum(taus)) <= 1e-15 * s * s                     # symmetric about 0
    if s == 1:
        assert taus == [0.]


# ---- the oracle's motion frame where nothing moves ----
def test_oracle_motion_frame_without_motion_is_the_lens_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    n = scene.num_prims
    v = np.tile([0.75, -0.5, 0.25], (n, 1))
    lens = lens_ref.render(oscene, 128, 96, 0., 1., 2, max_depth=4)["rgb"]
    assert np.array_equal(motion_ref.render(oscene, 128, 96, np.zeros((n, 3)), 2, max_depth=4)["rgb"], lens)
    one = lens_ref.render(oscene, 128, 96, 0., 1., 1, max_depth=4)["rgb"]
    assert np.array_equal(motion_ref.render(oscene, 128, 96, v, 1, max_depth=4)["rgb"], one)
    assert not np.array_equal(motion_ref.render(oscene, 128, 96, v, 2, max_depth=4)["rgb"], lens)


# ---- the motion kernel's per-ray code, compiled for the host, against the oracle's motion frame ----
# (scene, width, height, max_depth, workload options)
CASES = [("demo", 256, 160, 3, {}), ("stress", 160, 128, 6, dict(n_spheres=64, grid=7)),
         ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40))]
VIEWS = {"none": None, "yaw30": view_ref.VIEWS["yaw30"]}


def moving(scene, scale=1., seed=7):
    """One displacement per shape, seeded, in multiples of 1/64 (exact in FP32), up to `scale` per component."""
    rng = np.random.default_rng(seed)
    v = np.round(rng.uniform(-scale, scale, size=(len(scene.shapes), 3)) * 64.) / 64.
    return motion_ref.per_prim(scene, v)


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw = request.param
    desc = workloads.describe(name, **kw)
    scene = workloads.build_scene(desc)
    return name, w, h, depth, moving(scene), scene, build_oracle_scene(desc)


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_fp32_motion_path_meets_the_parity_criterion(case, view, s):
    name, w, h, depth, v, scene, oscene = case
    b = _basis(VIEWS[view])
    ref = motion_ref.render(oscene, w, h, v, s, basis=b, max_depth=depth)
    got = motion_emu.render(scene, w, h, v, s, basis=b, max_depth=depth, cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    assert not np.array_equal(got, lens_emu.render(scene, w, h, 0., 1., s, basis=b, max_depth=depth, cull=False)["rgb"])


def test_fp32_motion_path_through_a_lens_meets_the_parity_criterion():
    desc = workloads.describe("demo")
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    v = moving(scene)
    b = _basis(VIEWS["yaw30"])
    ref = motion_ref.render(oscene, 256, 160, v, 3, basis=b, aperture=0.4, focus=12.)
    got = motion_emu.render(scene, 256, 160, v, 3, basis=b, aperture=0.4, focus=12., cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, 160)
    assert r["fragile_frac"] < 0.2, r
    assert not np.array_equal(got, lens_emu.render(scene, 256, 160, 0.4, 12., 3, basis=b, cull=False)["rgb"])


BIT_CASES = [("demo", {}), ("cornell_box", {}), ("stress", dict(n_spheres=64, grid=7)), ("ngons", dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_swept_hierarchy_without_motion_is_the_scene_hierarchy(name, kw):
    scene = workloads.scene(name, **kw)
    nodes, prims, _ = emu.bvh(scene)
    sn, sp = motion_emu.swept_bvh(scene, np.zeros((scene.num_prims, 3)))
    assert sn.tobytes() == nodes.tobytes() and sp.tobytes() == prims.tobytes()
    mn, mp = motion_emu.swept_bvh(scene, moving(scene))
    assert mn.tobytes() != nodes.tobytes()


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_hierarchy_changes_no_pixel_of_a_moving_scene(name, kw):
    scene = workloads.scene(name, **kw)
    v = moving(scene, 2.)
    a = motion_emu.render(scene, 160, 96, v, 3, basis=_basis(VIEWS["yaw30"]), max_depth=4)["rgb"]
    c = motion_emu.render(scene, 160, 96, v, 3, basis=_basis(VIEWS["yaw30"]), max_depth=4, accel=True)["rgb"]
    assert np.array_equal(a, c)


# ---- a mover that can never be hit: the motion code is the lens code bit for bit ----
MATTE = dict(diffusion=1., diffuse_color=(0.7, 0.6, 0.5), specular=0.3, specular_exponent=30., is_glass_like=False, reflection=0.,
             refractive_index=1.)


def unhittable_mover():
    """The stress scene plus a clockwise-projected quad and triangle (never hit, culled or not) that move, the rest at rest."""
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    desc["polygons"] = list(desc.get("polygons", [])) + [([(-5., -5., -20.), (-5., 5., -20.), (5., 5., -20.), (5., -5., -20.)], MATTE),
                                                 ([(-8., -2., -25.), (-8., 4., -25.), (-2., 4., -25.)], MATTE)]
    scene = workloads.build_scene(desc)
    v = np.zeros((scene.num_prims, 3))
    k = len(desc["spheres"]) + len(desc["polygons"])            # shapes: spheres, polygons, meshes
    offs = np.cumsum([0] + [s.triangles.shape[0] if isinstance(s, Obj) else 1 for s in scene.shapes])
    for shape in (k - 2, k - 1):
        v[offs[shape]] = (3.5, -1.25, 2.)
    return scene, v


@pytest.mark.parametrize("cull", [True, False])
def test_an_unhittable_mover_leaves_the_lens_frame_bit_for_bit(cull):
    scene, v = unhittable_mover()
    assert np.abs(v).sum() > 0
    b = _basis(VIEWS["yaw30"])
    for accel in (False, True):
        got = motion_emu.render(scene, 160, 96, v, 3, basis=b, max_depth=5, cull=cull, accel=accel)["rgb"]
        want = lens_emu.render(scene, 160, 96, 0., 1., 3, basis=b, max_depth=5, cull=cull, accel=accel)["rgb"]
        assert got.tobytes() == want.tobytes() and got.any(), (cull, accel)


# ---- smear: a sphere moving sideways before a wall of stripes ----
CENTRE, RADIUS = np.array([0., 0., -12.]), 3.


def stripe_scene():
    stripes = []
    for k in range(-12, 12):
        x0, x1 = 1.5 * k, 1.5 * (k + 1)
        refl = dict(MATTE, diffuse_color=(0.9, 0.9, 0.9) if k % 2 else (0.05, 0.05, 0.05), specular=0.)
        stripes.append(([(x0, -20., -30.), (x1, -20., -30.), (x1, 20., -30.), (x0, 20., -30.)], refl))      # CCW: normal +z
    ball = dict(MATTE, diffuse_color=(0.2, 0.4, 0.9), specular=0.5, specular_exponent=50.)
    # the light at the camera: a wall point is in the ball's shadow exactly where the camera sees the ball in front of it
    desc = {"name": "stripes", "default": False, "spheres": [(tuple(CENTRE), RADIUS, ball)], "polygons": stripes, "meshes": [],
            "lights": [((0., 0., 0.), (1., 1., 1.), 1.)]}
    return workloads.build_scene(desc)


def _misses_swept_ball(w, h, s, v, fov=1.5):
    """(h, w): every pinhole sample ray of the pixel passes the ball's whole path [c - v/2, c + v/2] by more than 2 % of the
    radius."""
    hf = np.tan(fov / 2.)
    W, H = float(s * w), float(s * h)
    y, x, i, j = np.meshgrid(np.arange(h), np.arange(w), np.arange(s), np.arange(s), indexing="ij")
    d = np.stack([2. * ((s * x + j) / W - 0.5) * hf * (W / H), -2. * ((s * y + i) / H - 0.5) * hf, -np.ones(x.shape)], axis=-1)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    far = np.ones(d.shape[:-1], dtype=bool)
    for u in np.linspace(-0.5, 0.5, 401):
        c = CENTRE + u * np.asarray(v)
        tca = d @ c
        far &= np.sqrt(np.maximum(c @ c - tca * tca, 0.)) > 1.02 * RADIUS
    return far.all(axis=(2, 3))


def test_a_moving_ball_smears_along_its_path_and_nowhere_else():
    scene, w, h, s = stripe_scene(), 192, 160, 4
    lens = lens_emu.render(scene, w, h, 0., 1., s)["rgb"]
    extents = []
    for a in (0., 1., 2., 4.):
        v = motion_ref.per_prim(scene, [[a, 0., 0.]] + [[0., 0., 0.]] * (len(scene.shapes) - 1))
        f = motion_emu.render(scene, w, h, v, s)["rgb"]
        outside = _misses_swept_ball(w, h, s, (a, 0., 0.))
        assert outside.sum() > 10000
        assert f[outside].tobytes() == lens[outside].tobytes(), a
        changed = (f != lens).any(axis=2)
        extents.append(int(changed.any(axis=0).sum()))          # columns the smear reaches
    assert extents[0] == 0 and extents[1] < extents[2] < extents[3], extents


# ---- argument checks of the C ABI and of the Python mirror ----
def _motion(n=4, v=0.5, samples=2, null=False):
    arr = np.full((max(n, 1), 3), v, dtype=np.float64)
    m = _abi.RmMotion()
    m.n_prims, m.samples = n, samples
    m.displacement = None if null else arr.ctypes.data_as(C.POINTER(C.c_double))
    return m, arr


def _call(params=None, view=None, lens=None, motion=None, rgb=True, rgb8=False):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    return L.rm_render_motion(1, C.byref(p), C.byref(view) if view is not None else None, C.byref(lens) if lens is not None else None,
                              C.byref(motion) if motion is not None else None, out.ctypes.data if rgb else None,
                              out8.ctypes.data if rgb8 else None, None)


@pytest.mark.parametrize("kw", [None, dict(n=-1), dict(null=True), dict(v=np.nan), dict(v=np.inf), dict(v=-np.inf), dict(samples=0),
                                dict(samples=9)])
def test_invalid_motion_is_rejected(kw):
    if kw is None:
        assert _call(motion=None) == INVALID
        return
    m, _keep = _motion(**kw)
    assert _call(motion=m) == INVALID


def test_invalid_views_lenses_and_parameters_are_rejected():
    L = _abi.load()
    m, _keep = _motion()
    bad = _abi.RmView()
    bad.forward[:] = [0., 1., 0.]
    bad.up[:] = [0., 2., 0.]
    assert _call(view=bad, motion=m) == INVALID
    for ln in ((-0.1, 10., 2), (0.5, 0., 2), (np.nan, 10., 2), (0.5, 10., 3)):     # the last: lens->samples != motion->samples
        assert _call(lens=lens_emu.lens(*ln), motion=m) == INVALID, ln
    assert _call(motion=m, rgb=False) == INVALID
    for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
        setattr(p, field, value)
        assert _call(params=p, motion=m) == INVALID, field
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 48, 64)
    assert _call(params=p, motion=m) == DIMENSIONS
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 9024, 64)                  # the 8 x frame is wider than 65535
    m8, _keep8 = _motion(samples=8)
    assert _call(params=p, motion=m8) == DIMENSIONS


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    m, _keep = _motion()
    assert _call(motion=m) == NOT_INITIALISED
    assert _call(motion=m, lens=lens_emu.lens(0.5, 10., 2)) == NOT_INITIALISED
    m0, _keep0 = _motion(n=0, null=True)
    assert _call(motion=m0) == NOT_INITIALISED


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(displacement=[np.nan, 0., 0.]),
                                dict(displacement=[0., np.inf, 0.]), dict(displacement=[0.1, 0.2]), dict(displacement=[[1., 0., 0.]] * 2),
                                dict(aperture=-1.), dict(focus=0.), dict(forward=(0., 1., 0.), up=(0., 1., 0.))])
def test_renderer_rejects_invalid_motion_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(displacement=(0.5, 0., 0.))
    args.update(kw)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_motion(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **args)
