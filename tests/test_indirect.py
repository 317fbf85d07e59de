"""Diffuse interreflection (rm_render_indirect, include/rm_b200.h) without a GPU: the strata, disc points and bounce directions of
the shared definition code (rm::diffuse_offset, rm::diffuse_dir) against Python and the oracle's restatement bit for bit, the
oracle's indirect frame against its lens frame and against a closed form, and the indirect kernel's per-ray code compiled for
the host (tests/emu/rm_indirect_emu.cpp) against the oracle and against the lens kernel's.  GPU part:
tests/test_zz_indirect_gpu.py."""
import ctypes as C
import math

import numpy as np
import pytest

from rusty_marcher_b200 import _abi, workloads
from tests import indirect_ref, lens_ref, supersample_ref, view_ref
from tests.conftest import has_gpu
from tests.emu import indirect_emu, lens_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID, DIMENSIONS = -2, -3, -4            # include/rm_b200.h status codes


# ---- the strata and the disc points ----
@pytest.mark.parametrize("s", range(1, 9))
def test_diffuse_offset_is_the_python_and_oracle_definition_and_a_bijection(s):
    for level in range(1, 9):
        strata, points = set(), set()
        for i in range(s):
            for j in range(s):
                got = indirect_emu.diffuse_offset(s, i, j, level)
                assert got == indirect_ref.python_diffuse_offset(s, i, j, level) == indirect_ref.oracle_diffuse_offset(s, i, j, level)
                assert got[0] * got[0] + got[1] * got[1] < 1.
                strata.add(indirect_ref.stratum(s, i, j, level))
                points.add(got)
        assert len(strata) == len(points) == s * s, (s, level)
    if s == 1:
        assert indirect_emu.diffuse_offset(1, 0, 0, 1) == (0., 0.)


# coordinate functions of (i, j, L) of every stratified dimension: sub-pixel, lens, rough, area, time
OTHER_STRATA = [lambda i, j, L: i, lambda i, j, L: j, lambda i, j, L: i + j, lambda i, j, L: i + j + L, lambda i, j, L: i + 2 * j + L,
                lambda i, j, L: i + 3 * j, lambda i, j, L: 2 * i + j]


@pytest.mark.parametrize("s", range(4, 9))
def test_diffuse_strata_are_no_shifted_copy_of_another_dimension(s):
    i, j = np.meshgrid(np.arange(s), np.arange(s), indexing="ij")
    for level in range(1, 9):
        a, b = (np.array(x) for x in zip(*[indirect_ref.stratum(s, int(ii), int(jj), level) for ii, jj in zip(i.ravel(), j.ravel())]))
        for mine in (a, b):
            for other in OTHER_STRATA:
                diff = (mine - other(i, j, level).ravel()) % s
                assert len(set(diff.tolist())) > 1, (s, level)
        assert len(set(((a - b) % s).tolist())) > 1


def test_concentric_map_is_equal_area():
    s = 256
    pts = np.array([indirect_emu.diffuse_offset(s, i, j, 1) for i in range(s) for j in range(s)])
    r2 = pts[:, 0] ** 2 + pts[:, 1] ** 2
    assert r2.max() < 1.
    assert abs(r2.mean() - 0.5) < 1e-3
    assert abs(np.sqrt(1. - r2).mean() - 2. / 3.) < 1e-3
    # the elliptical grid map of lens_offset is not equal-area: Malley's lift of its points would not be cosine-weighted
    q = (2. * np.arange(s) + 1.) / s - 1.
    p, qq = np.meshgrid(q, q, indexing="ij")
    e2 = (p * np.sqrt(1. - qq * qq / 2.)) ** 2 + (qq * np.sqrt(1. - p * p / 2.)) ** 2
    assert abs(np.sqrt(1. - e2).mean() - 2. / 3.) > 0.03


# ---- the bounce direction and origin ----
def _normals():
    rng = np.random.default_rng(20261022)
    special = [(0., 0., 1.), (0., 0., -1.), (1., 0., 0.), (-1., 0., 0.), (0., 1., 0.), (0., -1., 0.), (0.6, 0.8, 0.), (0., -0.6, 0.8),
               (-0.8, 0., -0.6)]
    out = [np.array(n) for n in special]
    for _ in range(40):
        v = rng.normal(size=3)
        out.append(v / np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]))
    return out


@pytest.mark.parametrize("s", [1, 2, 3, 4, 8])
def test_diffuse_dir_is_unit_in_the_facing_hemisphere_and_the_oracle_definition(s):
    p = np.array([1., -2., 3.])
    for n in _normals():
        for incoming in (-n, n):                                # from the front and from behind: the normal turns against d
            nf = n if float(np.dot(n, incoming)) < 0. else -n
            for i in range(s):
                for j in range(s):
                    lx, ly = indirect_emu.diffuse_offset(s, i, j, 1 + (i + j) % 8)
                    o, rd = indirect_emu.diffuse_ray(p, n, incoming, lx, ly)
                    assert abs(float(np.dot(rd, rd)) - 1.) <= 1e-15
                    assert float(np.dot(rd, nf)) > 0., (n, incoming, lx, ly)
                    assert np.array_equal(rd, indirect_ref.oracle_diffuse_dir(nf, lx, ly))
                    assert np.array_equal(o, p + nf * 1e-4)
    _o, rd = indirect_emu.diffuse_ray(p, [0., 0., 1.], [0., 0., -1.], 0., 0.)
    assert np.array_equal(rd, [0., 0., 1.])                     # s = 1: along n_f


# ---- the oracle's indirect frame ----
def test_oracle_frame_without_bounces_is_the_lens_frame():
    desc = workloads.describe("stress", n_spheres=64, grid=7)
    oscene = build_oracle_scene(desc)
    for depth in (1, 4):
        lens = lens_ref.render(oscene, 128, 96, 0., 1., 2, max_depth=depth)["rgb"]
        got = indirect_ref.render(oscene, 128, 96, 2, max_depth=depth)["rgb"]
        assert np.array_equal(got, lens) == (depth == 1), depth
    black = indirect_ref.anchor_desc(with_target=False)
    ob = build_oracle_scene(black)
    assert np.array_equal(indirect_ref.render(ob, 128, 96, 3, max_depth=4)["rgb"], lens_ref.render(ob, 128, 96, 0., 1., 3, max_depth=4)["rgb"])


# ---- the furnace: the camera inside a diffuse sphere, lit by nothing but the background ----
@pytest.mark.parametrize("depth", [2, 3, 4, 5])
def test_furnace_closed_form(depth):
    rho = 0.6
    desc = indirect_ref.furnace_desc(rho)
    want = indirect_ref.furnace_value(rho, depth)
    ref = indirect_ref.render(build_oracle_scene(desc), 64, 64, 3, max_depth=depth)["rgb"]
    assert np.abs(ref / want - 1.).max() <= 1e-12
    got = indirect_emu.render(workloads.build_scene(desc), 64, 64, 3, max_depth=depth)["rgb"].astype(np.float64)
    assert np.abs(got / want - 1.).max() <= 1e-6


# ---- colour bleeding: a red sphere before a white wall ----
CENTRE, RADIUS = indirect_ref.BLEED_CENTRE, indirect_ref.BLEED_RADIUS


def _wall_pixels(w, h, fov=1.5):
    """(h, w) bool: the pinhole ray through the pixel's centre misses the sphere by 15 % of its radius (so every sub-pixel ray
    sees the wall); (h, w) distance of the pixel's wall point from the sphere's foot on the wall."""
    hf = np.tan(fov / 2.)
    y, x = np.meshgrid(np.arange(h) + 0.5, np.arange(w) + 0.5, indexing="ij")
    d = np.stack([2. * (x / w - 0.5) * hf * (w / h), -2. * (y / h - 0.5) * hf, -np.ones(x.shape)], axis=-1)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    c = np.array(CENTRE)
    tca = d @ c
    miss = np.sqrt(np.maximum(c @ c - tca * tca, 0.)) > 1.15 * RADIUS
    wall = d * (-30. / d[..., 2:3])
    return miss, np.hypot(wall[..., 0] - c[0], wall[..., 1] - c[1])


def test_red_sphere_bleeds_onto_the_white_wall():
    desc, w, h, s = indirect_ref.bleed_desc(), 192, 160, 4
    scene = workloads.build_scene(desc)
    miss, dist = _wall_pixels(w, h)
    lens = lens_emu.render(scene, w, h, 0., 1., s)["rgb"].astype(np.float64)
    assert np.array_equal(lens[..., 0][miss], lens[..., 1][miss])             # white light on a white wall: R = G everywhere
    ind = indirect_emu.render(scene, w, h, s, max_depth=3)["rgb"].astype(np.float64)
    rg = (ind[..., 0] - ind[..., 1])[miss]
    dm = dist[miss]
    rings = [rg[(dm >= a) & (dm < b)].mean() for a, b in ((3., 5.), (5., 8.), (8., 12.), (12., 18.))]
    assert rings[0] > rings[1] > rings[2] > rings[3] >= 0., rings
    assert rg.min() >= 0.                                       # only red light is added
    ref = indirect_ref.render(build_oracle_scene(desc), w, h, s, max_depth=3)
    lens_ref.check_parity(ind.astype(np.float32), _rgb8(ind.astype(np.float32)), ref, h)


# ---- the indirect kernel's per-ray code, compiled for the host, against the oracle's indirect frame ----
# (scene, width, height, max_depth, workload options)
CASES = [("demo", 192, 128, 3, {}), ("stress", 128, 96, 4, dict(n_spheres=64, grid=7)),
         ("ngons", 128, 96, 4, dict(n_spheres=12, n_polygons=40)), ("cornell_box", 128, 96, 3, {})]
VIEWS = {"none": None, "yaw30": view_ref.VIEWS["yaw30"]}


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, workloads.build_scene(desc), build_oracle_scene(desc)


def _basis(view):
    return None if view is None else view_ref.numpy_basis(*view)


def _rgb8(rgb):
    return supersample_ref.rgb8_of(rgb, rgb.max())


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("view", list(VIEWS), ids=list(VIEWS))
def test_fp32_indirect_path_meets_the_parity_criterion(case, view, s):
    name, w, h, depth, scene, oscene = case
    b = _basis(VIEWS[view])
    ref = indirect_ref.render(oscene, w, h, s, basis=b, max_depth=depth)
    got = indirect_emu.render(scene, w, h, s, basis=b, max_depth=depth, cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    assert not np.array_equal(got, lens_emu.render(scene, w, h, 0., 1., s, basis=b, max_depth=depth, cull=False)["rgb"])


def test_fp32_indirect_path_through_a_lens_meets_the_parity_criterion():
    desc = workloads.describe("demo")
    scene, oscene = workloads.build_scene(desc), build_oracle_scene(desc)
    b = _basis(VIEWS["yaw30"])
    ref = indirect_ref.render(oscene, 192, 128, 3, basis=b, aperture=0.4, focus=12.)
    got = indirect_emu.render(scene, 192, 128, 3, basis=b, aperture=0.4, focus=12., cull=False)["rgb"]
    r = lens_ref.check_parity(got, _rgb8(got), ref, 128)
    assert r["fragile_frac"] < 0.2, r


BIT_CASES = [("demo", {}), ("cornell_box", {}), ("stress", dict(n_spheres=64, grid=7)), ("ngons", dict(n_spheres=12, n_polygons=40))]


@pytest.mark.parametrize("name,kw", BIT_CASES, ids=[c[0] for c in BIT_CASES])
def test_hierarchy_changes_no_pixel(name, kw):
    scene = workloads.scene(name, **kw)
    a = indirect_emu.render(scene, 128, 96, 2, basis=_basis(VIEWS["yaw30"]), max_depth=4)["rgb"]
    c = indirect_emu.render(scene, 128, 96, 2, basis=_basis(VIEWS["yaw30"]), max_depth=4, accel=True)["rgb"]
    assert np.array_equal(a, c)


# ---- the never-hit anchor: black opaque surfaces and one diffuse triangle no ray can reach ----
@pytest.mark.parametrize("spheres", [True, False], ids=["spheres", "planes"])
def test_never_hit_diffuse_triangle_leaves_the_lens_frame(spheres):
    scene = workloads.build_scene(indirect_ref.anchor_desc(spheres=spheres))
    for accel in (False, True):
        for s, aperture in ((1, 0.), (3, 0.3)):
            want = lens_emu.render(scene, 128, 96, aperture, 20., s, max_depth=4, cull=False, accel=accel)
            got = indirect_emu.render(scene, 128, 96, s, aperture=aperture, focus=20., max_depth=4, cull=False, accel=accel)
            assert got["glass_mode"] == want["glass_mode"] and (spheres or got["glass_mode"] == 0)
            assert np.array_equal(got["rgb"], want["rgb"]), (accel, s)
    assert (want["rgb"] > 0.).any(axis=2).mean() > 0.3         # the black surfaces fill most of the frame


# ---- argument checks of the C ABI and of the Python mirror ----
def _call(params=None, view=None, lens=None, samples=2, rgb=True, rgb8=False):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    return L.rm_render_indirect(1, C.byref(p), C.byref(view) if view is not None else None, C.byref(lens) if lens is not None else None,
                                samples, out.ctypes.data if rgb else None, out8.ctypes.data if rgb8 else None, None)


def test_invalid_arguments_are_rejected():
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
    assert _call(params=p, samples=8) == DIMENSIONS


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    assert _call() == NOT_INITIALISED
    assert _call(lens=lens_emu.lens(0.5, 10., 2)) == NOT_INITIALISED
    assert _call(samples=1, rgb=False, rgb8=True) == NOT_INITIALISED


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(samples=True), dict(aperture=-1.),
                                dict(focus=0.), dict(aperture=math.nan), dict(forward=(0., 1., 0.), up=(0., 1., 0.)),
                                dict(patch_rows=(0, -1, 2))])
def test_renderer_rejects_invalid_indirect_arguments(kw):
    import rusty_marcher_b200 as rm
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_indirect(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **kw)
