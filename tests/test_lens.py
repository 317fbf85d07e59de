"""Depth of field (rm_render_lens, include/rm_b200.h RmLens) without a GPU: the lens points and sample rays of the shared
definition code (rm::lens_offset, rm::lens_ray) against numpy and the oracle's restatement bit for bit, the oracle's lens
frame against the supersampled definition, and the lens kernel's per-ray code compiled for the host (tests/emu/rm_lens_emu.cpp)
against the oracle.  GPU part: tests/test_zz_lens_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi, workloads
from tests import lens_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import lens_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


@pytest.mark.parametrize("s", range(1, 9))
def test_lens_offset_is_the_numpy_definition_and_lies_in_the_unit_disc(s):
    strata = set()
    for i in range(s):
        for j in range(s):
            lx, ly = lens_emu.lens_offset(s, i, j)
            nx, ny = lens_ref.numpy_lens_offset(s, i, j)
            ox, oy = lens_ref.oracle_lens_offset(s, i, j)
            assert (lx, ly) == (nx, ny) == (ox, oy), (s, i, j)
            assert lx * lx + ly * ly <= 1.
            strata.add(((i + j) % s, j))
    assert len(strata) == s * s                                  # (i, j) -> (a, b) is a bijection of the s x s strata
    if s == 1:
        assert lens_emu.lens_offset(1, 0, 0) == (0., 0.)       # s = 1: the lens centre only


def _ray_cases():
    rng = np.random.default_rng(20261021)
    views = [None] + [view_ref.numpy_basis(*v) for v in view_ref.VIEWS.values()]
    cases = []
    for k in range(1000):
        w, h = 32 * int(rng.integers(1, 9)), int(rng.integers(16, 300))
        s = int(rng.integers(1, 9))
        aperture = 0. if k % 10 == 0 else float(10. ** rng.uniform(-3, 1.5))
        if k % 7 == 3:                                          # a random valid view
            b = None
            while b is None:
                b = view_ref.numpy_basis(tuple(rng.normal(size=3)), tuple(rng.normal(size=3)))
        else:
            b = views[k % len(views)]
        cases.append((tuple(rng.normal(size=3) * 10. ** rng.uniform(-2, 2.5)), w, h, float(rng.uniform(0.2, 2.8)), b, aperture,
                      float(10. ** rng.uniform(-1, 3)), s, int(rng.integers(0, w)), int(rng.integers(0, h)),
                      int(rng.integers(0, s)), int(rng.integers(0, s))))
    return cases


def test_lens_ray_equals_the_oracle_restatement_bit_for_bit():
    for case in _ray_cases():
        o, d = lens_emu.lens_ray(*case)
        ro, rd = lens_ref.oracle_lens_ray(*case)
        assert np.array_equal(o, ro) and np.array_equal(d, rd), case


def test_aperture_zero_rays_are_the_pinhole_rays():
    o, d = lens_emu.lens_ray((1., 2., 3.), 160, 128, 1.5, None, 0., 10., 4, 17, 33, 2, 3)
    assert o.tolist() == [1., 2., 3.]
    a, b = lens_emu.lens_ray((1., 2., 3.), 160, 128, 1.5, None, 0.5, 10., 1, 17, 33, 0, 0)
    assert a.tolist() == [1., 2., 3.]                            # s = 1: the lens centre
    assert np.allclose(b, lens_emu.lens_ray((1., 2., 3.), 160, 128, 1.5, None, 0., 10., 1, 17, 33, 0, 0)[1], rtol=0, atol=1e-15)


def test_oracle_lens_without_aperture_is_the_supersampled_frame():
    scene = O.Scene.create_default()
    for s in (1, 2, 3):
        got = lens_ref.render(scene, 160, 128, 0., 10., s)["rgb"]
        want = supersample_ref.render_supersampled(scene, 160, 128, s)["rgb"]
        assert np.array_equal(got, want), s


# ---- the lens kernel's per-ray code, compiled for the host, against the oracle's lens frame ----
# (scene, width, height, max_depth, workload options, focus, aperture)
CASES = [("demo", 256, 160, 3, {}, 12., 0.4), ("cornell_box", 160, 128, 3, {}, 300., 8.),
         ("stress", 160, 128, 6, dict(n_spheres=64, grid=7), 120., 2.),
         ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40), 30., 0.6)]
VIEWS = {"none": None, "yaw30": view_ref.VIEWS["yaw30"]}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw, focus, aperture = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, focus, aperture, workloads.build_scene(desc), build_oracle_scene(desc)


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_fp32_lens_path_meets_the_parity_criterion(case, view, s):
    name, w, h, depth, focus, aperture, scene, oscene = case
    b = _basis(VIEWS[view])
    ref = lens_ref.render(oscene, w, h, aperture, focus, s, basis=b, max_depth=depth)
    got = lens_emu.render(scene, w, h, aperture, focus, s, basis=b, max_depth=depth, cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    assert got.any() or (name == "cornell_box" and view == "yaw30")


@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_hierarchy_changes_no_pixel(case, view):
    name, w, h, depth, focus, aperture, scene, _ = case
    b = _basis(VIEWS[view])
    a = lens_emu.render(scene, w, h, aperture, focus, 2, basis=b, max_depth=depth)["rgb"]
    c = lens_emu.render(scene, w, h, aperture, focus, 2, basis=b, max_depth=depth, accel=True)["rgb"]
    assert np.array_equal(a, c)


def _focal_scene(focus, sphere=True):
    """A diffuse quad facing the camera at distance `focus`, and a sphere farther away beside it, lit by the default lights."""
    matte = dict(diffusion=1., diffuse_color=(0.7, 0.6, 0.5), specular=0., specular_exponent=30., is_glass_like=False,
                 reflection=0.95, refractive_index=1.)
    quad = [(-6., -4., -focus), (6., -4., -focus), (6., 4., -focus), (-6., 4., -focus)]       # CCW in XY: normal +z
    spheres = [((2. * focus, 1.2 * focus, -3. * focus), 2., matte)] if sphere else []
    desc = {"name": "focal", "default": False, "spheres": spheres, "polygons": [(quad, matte)],
            "meshes": [], "lights": workloads.DEFAULT_LIGHTS}
    return workloads.build_scene(desc)


def test_the_plane_in_focus_stays_sharp():
    focus, w, h = 10., 160, 128
    scene = _focal_scene(focus)
    pin = lens_emu.render(scene, w, h, 0., focus, 4)["rgb"]
    lens = lens_emu.render(scene, w, h, 1.5, focus, 4)["rgb"]
    # the quad's interior: pixels whose 5 x 5 neighbourhood lies inside it, from the pinhole frame of the quad alone
    hit = np.all(lens_emu.render(_focal_scene(focus, sphere=False), w, h, 0., focus, 4)["rgb"] > 0.1 + 1e-3, axis=2)
    inner = hit.copy()
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            inner &= np.roll(np.roll(hit, dy, 0), dx, 1)
    assert inner.sum() > 2000
    rel = np.abs(lens[inner].astype(np.float64) - pin[inner]) / np.abs(pin[inner])
    assert rel.max() <= 1e-4, rel.max()
    assert not np.array_equal(lens, pin)                         # the sphere behind it is blurred


def test_more_aperture_blurs_more_pixels():
    scene = workloads.scene("demo")
    pin = lens_emu.render(scene, 160, 128, 0., 12., 3)["rgb"]
    shares = []
    for a in (0.05, 0.3, 1.5):
        lens = lens_emu.render(scene, 160, 128, a, 12., 3)["rgb"]
        shares.append(float((np.abs(lens - pin).max(axis=2) > 1e-3 * np.maximum(pin.max(axis=2), 1e-3)).mean()))
    assert shares[0] < shares[1] < shares[2], shares


# ---- argument checks of the C ABI and of the Python mirror ----
def _call(params=None, view=None, lens=None, rgb=True, rgb8=False):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    return L.rm_render_lens(1, C.byref(p), C.byref(view) if view is not None else None, C.byref(lens) if lens is not None else None,
                            out.ctypes.data if rgb else None, out8.ctypes.data if rgb8 else None, None)


def _lens(aperture=0.5, focus=10., samples=2):
    return lens_emu.lens(aperture, focus, samples)


@pytest.mark.parametrize("lens", [None, (0.5, 10., 0), (0.5, 10., 9), (-0.1, 10., 2), (0.5, 0., 2), (0.5, -1., 2),
                                  (np.nan, 10., 2), (np.inf, 10., 2), (0.5, np.inf, 2), (0.5, np.nan, 2)])
def test_invalid_lenses_are_rejected(lens):
    assert _call(lens=None if lens is None else _lens(*lens)) == INVALID


def test_invalid_views_and_parameters_are_rejected():
    L = _abi.load()
    bad = _abi.RmView()
    bad.forward[:] = [0., 1., 0.]
    bad.up[:] = [0., 2., 0.]
    assert _call(view=bad, lens=_lens()) == INVALID
    assert _call(lens=_lens(), rgb=False) == INVALID
    for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
        setattr(p, field, value)
        assert _call(params=p, lens=_lens()) == INVALID, field
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 48, 64)
    assert _call(params=p, lens=_lens()) == DIMENSIONS
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 9024, 64)                  # the 8 x frame is wider than 65535
    assert _call(params=p, lens=_lens(samples=8)) == DIMENSIONS


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    assert _call(lens=_lens()) == NOT_INITIALISED
    assert _call(lens=_lens(aperture=0.)) == NOT_INITIALISED     # (the pinhole frame: rm_render_supersampled)


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(aperture=-1.), dict(aperture=np.nan),
                                dict(focus=0.), dict(focus=np.inf), dict(forward=(0., 1., 0.), up=(0., 1., 0.))])
def test_renderer_rejects_invalid_lens_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(aperture=0.5, focus=10.)
    args.update(kw)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_lens(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **args)
