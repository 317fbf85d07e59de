"""Rough glass (rm_render_rough_glass, include/rm_b200.h RmRoughGlass) without a GPU: the turned direction and the strata of the
shared definition code (rm::rough_dir, rm::rough_offset) against numpy and the oracle's restatement bit for bit, the oracle's
rough frame against its lens frame where nothing turns, and the rough kernel's per-ray code compiled for the host
(tests/emu/rm_rough_emu.cpp) against the oracle and against the lens kernel's.  GPU part: tests/test_zz_rough_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import lens_ref, rough_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import lens_emu, rough_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


@pytest.mark.parametrize("s", range(1, 9))
def test_rough_offset_is_a_bijection_at_every_level(s):
    for level in range(1, 9):
        strata = set()
        for i in range(s):
            for j in range(s):
                got = rough_emu.rough_offset(s, i, j, level)
                assert got == rough_ref.oracle_rough_offset(s, i, j, level) == lens_ref.numpy_lens_offset(s, (j + level) % s, i)
                strata.add(got)
        assert len(strata) == s * s, (s, level)
    if s == 1:
        assert rough_emu.rough_offset(1, 0, 0, 1) == (0., 0.)


def _dir_cases():
    rng = np.random.default_rng(20261022)
    special = [(0., 0., 1.), (0., 0., -1.), (1., 0., 0.), (-1., 0., 0.), (0., 1., 0.), (0., -1., 0.), (0.6, 0.8, 0.), (0.6, 0.8, -0.),
               (0., -0.6, 0.8), (-0.8, 0., -0.6)]
    cases = []
    for k in range(1000):
        if k < 3 * len(special):
            rd = np.array(special[k % len(special)], dtype=np.float64)
        else:
            v = rng.normal(size=3)
            rd = v / np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
        g = 0. if k % 17 == 5 else float(10. ** rng.uniform(-4, 1))
        s = 1 + k % 8
        i, j, level = int(rng.integers(0, s)), int(rng.integers(0, s)), 1 + int(rng.integers(0, 8))
        cases.append((tuple(float(x) for x in rd), g, s, i, j, level))
    return cases


def test_rough_dir_is_the_numpy_and_oracle_definition_bit_for_bit():
    unchanged = turned = 0
    for rd, g, s, i, j, level in _dir_cases():
        lx, ly = rough_emu.rough_offset(s, i, j, level)
        got = rough_emu.rough_dir(rd, g, lx, ly)
        assert np.array_equal(got, rough_ref.numpy_rough_dir(rd, g, lx, ly)), (rd, g, s, i, j, level)
        assert np.array_equal(got, rough_ref.oracle_rough_dir(rd, g, lx, ly)), (rd, g, s, i, j, level)
        r = np.array(rd)
        if g == 0. or (lx == 0. and ly == 0.):
            assert np.array_equal(got, r)                        # bit for bit, -0 included
            assert all(np.signbit(got) == np.signbit(r))
            unchanged += 1
            continue
        turned += 1
        assert abs(float(np.dot(got, got)) - 1.) <= 1e-15
        angle = np.arctan2(np.linalg.norm(np.cross(r, got)), float(np.dot(r, got)))
        assert angle <= np.arctan(g) * (1. + 1e-12) + 1e-15, (rd, g, lx, ly, angle)
    assert unchanged > 50 and turned > 800


def test_turned_origins_follow_the_producing_function():
    p, n = np.array([1., 2., 3.]), np.array([0., 0., 1.])
    inc = np.array([0., 0.6, -0.8])                              # against the normal: refract_ray keeps n
    assert np.array_equal(rough_emu.rough_origin(0, p, n, inc, [0., 0., -1.]), p - n * 1e-4)
    assert np.array_equal(rough_emu.rough_origin(0, p, n, inc, [0., 0., 1.]), p + n * 1e-4)
    assert np.array_equal(rough_emu.rough_origin(1, p, n, inc, [0., 0.1, -0.99]), p - n * 1e-4)
    inside = np.array([0., 0.6, 0.8])                            # leaving through the surface: refract_ray turns n to -n
    assert np.array_equal(rough_emu.rough_origin(1, p, n, inside, [0., 0.1, 0.99]), p - (-n) * 1e-4)
    assert np.array_equal(rough_emu.rough_origin(1, p, n, inside, [0., 0.1, -0.99]), p + (-n) * 1e-4)


# ---- the oracle's rough frame where nothing turns ----
def test_oracle_rough_frame_without_turns_is_the_lens_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    n = scene.num_prims
    lens = lens_ref.render(oscene, 128, 96, 0., 1., 2, max_depth=4)["rgb"]
    assert np.array_equal(rough_ref.render(oscene, 128, 96, np.zeros(n), 2, max_depth=4)["rgb"], lens)
    opaque = np.where(rough_ref.glass_like(scene), 0., 0.5)
    assert opaque.any() and rough_ref.glass_like(scene).any()
    assert np.array_equal(rough_ref.render(oscene, 128, 96, opaque, 2, max_depth=4)["rgb"], lens)
    one = lens_ref.render(oscene, 128, 96, 0., 1., 1, max_depth=4)["rgb"]
    assert np.array_equal(rough_ref.render(oscene, 128, 96, np.full(n, 0.5), 1, max_depth=4)["rgb"], one)
    assert not np.array_equal(rough_ref.render(oscene, 128, 96, np.full(n, 0.5), 2, max_depth=4)["rgb"], lens)


# ---- the rough kernel's per-ray code, compiled for the host, against the oracle's rough frame ----
# (scene, width, height, max_depth, workload options, roughness of the glass-like primitives)
CASES = [("demo", 256, 160, 3, {}, 0.1), ("stress", 160, 128, 6, dict(n_spheres=64, grid=7), 0.05),
         ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40), 0.2)]
VIEWS = {"none": None, "yaw30": view_ref.VIEWS["yaw30"]}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw, g = request.param
    desc = workloads.describe(name, **kw)
    scene = workloads.build_scene(desc)
    return name, w, h, depth, np.where(rough_ref.glass_like(scene), g, 0.), scene, build_oracle_scene(desc)


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_fp32_rough_path_meets_the_parity_criterion(case, view, s):
    name, w, h, depth, g, scene, oscene = case
    b = _basis(VIEWS[view])
    ref = rough_ref.render(oscene, w, h, g, s, basis=b, max_depth=depth)
    got = rough_emu.render(scene, w, h, g, s, basis=b, max_depth=depth, cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    assert not np.array_equal(got, lens_emu.render(scene, w, h, 0., 1., s, basis=b, max_depth=depth, cull=False)["rgb"])


def test_fp32_rough_path_through_a_lens_meets_the_parity_criterion():
    desc = workloads.describe("demo")
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    g = np.where(rough_ref.glass_like(scene), 0.1, 0.)
    b = _basis(VIEWS["yaw30"])
    ref = rough_ref.render(oscene, 256, 160, g, 3, basis=b, aperture=0.4, focus=12.)
    got = rough_emu.render(scene, 256, 160, g, 3, basis=b, aperture=0.4, focus=12., cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, 160)
    assert r["fragile_frac"] < 0.2, r
    assert not np.array_equal(got, lens_emu.render(scene, 256, 160, 0.4, 12., 3, basis=b, cull=False)["rgb"])


BIT_CASES = [("demo", {}), ("cornell_box", {}), ("stress", dict(n_spheres=64, grid=7)), ("ngons", dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_rough_code_without_roughness_is_the_lens_code_bit_for_bit(name, kw):
    scene = workloads.scene(name, **kw)
    b = _basis(VIEWS["yaw30"])
    for basis, aperture in ((None, 0.), (b, 0.3)):
        want = lens_emu.render(scene, 160, 96, aperture, 20., 3, basis=basis, max_depth=4)["rgb"]
        got = rough_emu.render(scene, 160, 96, np.zeros(scene.num_prims), 3, basis=basis, aperture=aperture, focus=20., max_depth=4)["rgb"]
        assert np.array_equal(got, want), (name, aperture)


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_hierarchy_changes_no_pixel(name, kw):
    scene = workloads.scene(name, **kw)
    g = np.full(scene.num_prims, 0.15)
    a = rough_emu.render(scene, 160, 96, g, 2, basis=_basis(VIEWS["yaw30"]), max_depth=4)["rgb"]
    c = rough_emu.render(scene, 160, 96, g, 2, basis=_basis(VIEWS["yaw30"]), max_depth=4, accel=True)["rgb"]
    assert np.array_equal(a, c)


# ---- blur: a glass sphere in front of a wall of stripes ----
GLASS = dict(diffusion=0.1, diffuse_color=(1., 1., 1.), specular=0.5, specular_exponent=100., is_glass_like=True, reflection=0.1,
             refractive_index=1.5)
CENTRE, RADIUS = (0., 0., -12.), 3.


def stripe_scene():
    stripes = []
    for k in range(-12, 12):
        x0, x1 = 1.5 * k, 1.5 * (k + 1)
        refl = dict(diffusion=1., diffuse_color=(0.9, 0.9, 0.9) if k % 2 else (0.05, 0.05, 0.05), specular=0., specular_exponent=30.,
                    is_glass_like=False, reflection=0., refractive_index=1.)
        stripes.append(([(x0, -20., -30.), (x1, -20., -30.), (x1, 20., -30.), (x0, 20., -30.)], refl))      # CCW: normal +z
    desc = {"name": "stripes", "default": False, "spheres": [(CENTRE, RADIUS, GLASS)], "polygons": stripes, "meshes": [],
            "lights": [((0., 10., 5.), (1., 1., 1.), 1.)]}
    return workloads.build_scene(desc)


def _sample_hits_sphere(w, h, s, fov=1.5):
    """(h, w, s*s) bool: the pinhole sample ray meets the sphere, with a margin of 1 % of the radius either way (True where
    it surely does, and a second mask where it surely does not)."""
    hf = np.tan(fov / 2.)
    W, H = float(s * w), float(s * h)
    y, x, i, j = np.meshgrid(np.arange(h), np.arange(w), np.arange(s), np.arange(s), indexing="ij")
    d = np.stack([2. * ((s * x + j) / W - 0.5) * hf * (W / H), -2. * ((s * y + i) / H - 0.5) * hf, -np.ones(x.shape)], axis=-1)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    c = np.array(CENTRE)
    tca = d @ c
    dist = np.sqrt(np.maximum(c @ c - tca * tca, 0.))
    return (dist < 0.99 * RADIUS).reshape(h, w, s * s), (dist > 1.01 * RADIUS).reshape(h, w, s * s)


def test_roughness_blurs_what_the_glass_shows_and_nothing_else():
    scene, w, h, s = stripe_scene(), 192, 160, 4
    glass = rough_ref.glass_like(scene)
    hit, miss = _sample_hits_sphere(w, h, s)
    inside, outside = hit.all(axis=2), miss.all(axis=2)
    assert inside.sum() > 1000 and outside.sum() > 10000
    lens = lens_emu.render(scene, w, h, 0., 1., s)["rgb"]
    tvs = []
    for g in (0., 0.02, 0.1, 0.3):
        f = rough_emu.render(scene, w, h, np.where(glass, g, 0.), s)["rgb"].astype(np.float64)
        both_x, both_y = inside[:, 1:] & inside[:, :-1], inside[1:, :] & inside[:-1, :]
        tvs.append(float(np.abs(f[:, 1:] - f[:, :-1]).sum(axis=2)[both_x].sum() + np.abs(f[1:, :] - f[:-1, :]).sum(axis=2)[both_y].sum()))
        assert np.array_equal(f[outside], lens[outside].astype(np.float64)), g
    assert tvs[0] > tvs[1] > tvs[2] > tvs[3], tvs


# ---- argument checks of the C ABI and of the Python mirror ----
def _rough(n=4, g=0.1, samples=2, null=False):
    arr = np.full(max(n, 1), g, dtype=np.float64)
    r = _abi.RmRoughGlass()
    r.n_prims, r.samples = n, samples
    r.roughness = None if null else arr.ctypes.data_as(C.POINTER(C.c_double))
    return r, arr


def _call(params=None, view=None, lens=None, rough=None, rgb=True, rgb8=False):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    return L.rm_render_rough_glass(1, C.byref(p), C.byref(view) if view is not None else None, C.byref(lens) if lens is not None else None,
                                   C.byref(rough) if rough is not None else None, out.ctypes.data if rgb else None,
                                   out8.ctypes.data if rgb8 else None, None)


@pytest.mark.parametrize("kw", [None, dict(n=-1), dict(null=True), dict(g=-0.1), dict(g=np.nan), dict(g=np.inf), dict(samples=0),
                                dict(samples=9)])
def test_invalid_roughness_is_rejected(kw):
    if kw is None:
        assert _call(rough=None) == INVALID
        return
    r, _keep = _rough(**kw)
    assert _call(rough=r) == INVALID


def test_invalid_views_lenses_and_parameters_are_rejected():
    L = _abi.load()
    r, _keep = _rough()
    bad = _abi.RmView()
    bad.forward[:] = [0., 1., 0.]
    bad.up[:] = [0., 2., 0.]
    assert _call(view=bad, rough=r) == INVALID
    for ln in ((-0.1, 10., 2), (0.5, 0., 2), (np.nan, 10., 2), (0.5, 10., 3)):     # the last: lens->samples != rough->samples
        assert _call(lens=lens_emu.lens(*ln), rough=r) == INVALID, ln
    assert _call(rough=r, rgb=False) == INVALID
    for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
        setattr(p, field, value)
        assert _call(params=p, rough=r) == INVALID, field
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 48, 64)
    assert _call(params=p, rough=r) == DIMENSIONS
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 9024, 64)                  # the 8 x frame is wider than 65535
    r8, _keep8 = _rough(samples=8)
    assert _call(params=p, rough=r8) == DIMENSIONS


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    r, _keep = _rough()
    assert _call(rough=r) == NOT_INITIALISED
    assert _call(rough=r, lens=lens_emu.lens(0.5, 10., 2)) == NOT_INITIALISED
    r0, _keep0 = _rough(n=0, null=True)
    assert _call(rough=r0) == NOT_INITIALISED


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(roughness=-1.), dict(roughness=np.nan),
                                dict(roughness=[0.1, 0.2]), dict(roughness=np.inf), dict(aperture=-1.), dict(focus=0.),
                                dict(forward=(0., 1., 0.), up=(0., 1., 0.))])
def test_renderer_rejects_invalid_rough_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(roughness=0.1)
    args.update(kw)
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_rough_glass(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **args)
