"""Soft shadows (rm_render_area_lights, include/rm_b200.h RmAreaLights) without a GPU: the light frame and sample points of the
shared definition code (rm::light_frame, rm::light_sample) against numpy and the oracle's restatement bit for bit, the oracle's
area frame against its plain frame, and the area kernel's per-pixel code compiled for the host (tests/emu/rm_area_emu.cpp)
against the oracle.  GPU part: tests/test_zz_area_gpu.py."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi, workloads
from tests import area_ref, lens_ref, supersample_ref
from tests.conftest import has_gpu
from tests.emu import area_emu, emu, lens_emu
from tests.oracle_scenes import build_oracle_scene

NOT_INITIALISED, INVALID = -2, -3                           # include/rm_b200.h status codes


def _cases():
    rng = np.random.default_rng(20261021)
    out = []
    for k in range(1000):
        m = rng.normal(size=3)
        if k % 50 == 0:                                         # the branch-free formula's edge: m.z = +-0 and m = +-z
            m = [[0., 0., 1.], [0., 0., -1.], [1., 0., 0.], [0., 1., -0.], [0.6, 0.8, 0.]][k // 50 % 5]
        m = np.asarray(m, dtype=np.float64)
        m = m / np.sqrt(m @ m)
        c = rng.normal(size=3) * 10. ** rng.uniform(-1, 2.5)
        r = float(10. ** rng.uniform(-3, 1.5))
        s = int(rng.integers(1, 9))
        out.append((m, c, r, s, int(rng.integers(0, s)), int(rng.integers(0, s))))
    return out


def _ulp(x):
    return float(np.spacing(np.float64(abs(x))))


def test_light_frame_and_samples_equal_numpy_and_the_oracle_bit_for_bit():
    for m, c, r, s, a, b in _cases():
        t1, t2 = area_emu.light_frame(m)
        n1, n2 = area_ref.numpy_light_frame(m)
        o1, o2 = area_ref.oracle_light_frame(m)
        assert np.array_equal(t1, n1) and np.array_equal(t1, o1) and np.array_equal(t2, n2) and np.array_equal(t2, o2), m
        lx, ly = lens_emu.lens_offset(s, a, b)
        assert (lx, ly) == lens_ref.numpy_lens_offset(s, a, b)
        q = area_emu.light_sample(c, r, t1, t2, lx, ly)
        assert np.array_equal(q, area_ref.numpy_light_sample(c, r, t1, t2, lx, ly))
        assert np.array_equal(q, area_ref.oracle_light_sample(c, r, t1, t2, lx, ly)), (m, c, r, s, a, b)


def test_light_frame_is_orthonormal_and_samples_lie_on_the_facing_disc():
    for m, c, r, s, a, b in _cases():
        t1, t2 = area_emu.light_frame(m)
        for u, v, want in ((t1, t1, 1.), (t2, t2, 1.), (m, m, 1.), (t1, t2, 0.), (t1, m, 0.), (t2, m, 0.)):
            assert abs(float(u @ v) - want) <= 1e-15, (m, u, v)
        lx, ly = lens_emu.lens_offset(s, a, b)
        q = area_emu.light_sample(c, r, t1, t2, lx, ly)
        # exact offset q - c; q itself is rounded to the grid of c, hence the few ulp of |c| + r on top of the 1e-15
        d = [Fraction(float(q[k])) - Fraction(float(c[k])) for k in range(3)]
        slack = 2. * max(_ulp(abs(c[k]) + r) for k in range(3))
        norm = float(sum(x * x for x in d)) ** 0.5
        assert norm <= r * (1. + 1e-15) + 2. * slack, (norm, r)
        assert abs(float(sum(d[k] * Fraction(float(m[k])) for k in range(3)))) <= 1e-15 * r + 2. * slack
    # s = 1: the only point is the centre, exactly
    t1, t2 = area_emu.light_frame(np.array([0.6, 0., 0.8]))
    assert np.array_equal(area_emu.light_sample((1., 2., 3.), 5., t1, t2, *lens_emu.lens_offset(1, 0, 0)), [1., 2., 3.])


CASES = [("demo", 256, 160, 3, {}), ("cornell_box", 160, 128, 3, {}), ("stress", 160, 128, 6, dict(n_spheres=64, grid=7)),
         ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40))]
RADII = (0., 3.)                                                # the light at the camera stays a point, the other is a sphere


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, workloads.build_scene(desc), build_oracle_scene(desc)


def test_oracle_area_frame_is_the_plain_frame_at_one_sample_and_zero_radii(case):
    name, w, h, depth, _, oscene = case
    plain = O.render(oscene, w, h, max_depth=depth)
    for radii, s in ((RADII, 1), ((0., 0.), 3), ((2., 7.), 1)):
        got = area_ref.render(oscene, w, h, radii, s, max_depth=depth)
        assert np.array_equal(got["rgb"], plain["rgb"]), (radii, s)
        assert np.array_equal(got["prim_id"], plain["prim_id"])


@pytest.mark.parametrize("s", [2, 3, 4])
def test_fp32_area_path_meets_the_parity_criterion(case, s):
    name, w, h, depth, scene, oscene = case
    ref = area_ref.render(oscene, w, h, RADII, s, max_depth=depth)
    got = area_emu.render(scene, w, h, RADII, s, max_depth=depth, cull=False)
    r = lens_ref.check_parity(got["rgb"], supersample_ref.rgb8_of(got["rgb"], got["rgb"].max()), ref, (h // 32) * 32)
    assert r["fragile_frac"] < 0.2, r
    assert np.array_equal(got["prim_id"][ref["fragile"] & 1 == 0], ref["prim_id"][ref["fragile"] & 1 == 0])
    assert not np.array_equal(got["rgb"], emu.render(scene, w, h, "fast", max_depth=depth, cull=False)["rgb"])   # it does change


def test_hierarchy_changes_no_pixel(case):
    name, w, h, depth, scene, _ = case
    for s in (2, 3):
        a = area_emu.render(scene, w, h, RADII, s, max_depth=depth)
        c = area_emu.render(scene, w, h, RADII, s, max_depth=depth, accel=True)
        assert np.array_equal(a["rgb"], c["rgb"]) and np.array_equal(a["prim_id"], c["prim_id"]), s


def test_primary_ids_are_the_render_kernels(case):
    name, w, h, depth, scene, _ = case
    got = area_emu.render(scene, w, h, RADII, 2, max_depth=depth)
    assert np.array_equal(got["prim_id"], emu.render(scene, w, h, "fast", max_depth=depth)["prim_id"])


def _shadow_scene(occluder=True):
    """A diffuse wall facing the camera, one light in front of it and a sphere between them: a shadow whose edge the light's
    size softens."""
    matte = dict(diffusion=1., diffuse_color=(0.8, 0.8, 0.8), specular=0., specular_exponent=30., is_glass_like=False,
                 reflection=0.95, refractive_index=1.)
    quad = [(-12., -9., -20.), (12., -9., -20.), (12., 9., -20.), (-12., 9., -20.)]          # CCW in XY: normal +z
    spheres = [((3., -1.5, -13.), 1.5, matte)] if occluder else []
    desc = {"name": "shadow", "default": False, "spheres": spheres, "polygons": [(quad, matte)], "meshes": [],
            "lights": [((6., -3., -6.), (1., 1., 1.), 1.)]}
    return workloads.build_scene(desc)


def test_penumbra_grows_with_the_radius_and_a_tiny_light_is_the_point_light():
    scene, bare, w, h = _shadow_scene(), _shadow_scene(occluder=False), 160, 128
    point = emu.render(scene, w, h, "fast", cull=False)
    wall = point["prim_id"] == 1                               # the quad (the sphere is primitive 0)
    assert wall.sum() > 2000 and (wall & (point["rgb"].max(axis=2) <= 0.1 + 1e-6)).sum() > 100   # a hard shadow on it
    counts = []
    for radius in (0.3, 1., 2.5):
        v = area_emu.render(scene, w, h, [radius], 4, cull=False)["rgb"].max(axis=2)
        lit = area_emu.render(bare, w, h, [radius], 4, cull=False)["rgb"].max(axis=2)     # the same light, nothing in the way
        partial = wall & (v > 0.1 + 1e-4) & (v < lit * (1. - 1e-4))      # strictly between fully shadowed and fully lit
        counts.append(int(partial.sum()))
    assert counts[0] < counts[1] < counts[2], counts
    tiny = area_emu.render(scene, w, h, [1e-6], 4, cull=False)["rgb"]
    assert np.abs(tiny.astype(np.float64) - point["rgb"]).max() <= 1e-4


# ---- argument checks of the C ABI and of the Python mirror ----
def _call(params=None, lights=None, rgb=True, rgb8=False, handle=1):
    L = _abi.load()
    p = params
    if p is None:
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    out8 = np.zeros((64, 64, 3), dtype=np.uint8)
    return L.rm_render_area_lights(handle, C.byref(p), C.byref(lights) if lights is not None else None, out.ctypes.data if rgb else None,
                                   None, out8.ctypes.data if rgb8 else None, None)


_keep = []


def _lights(radii=(0., 1.), samples=2, n=None, null_radius=False):
    a = (C.c_double * max(len(radii), 1))(*radii)
    _keep.append(a)
    al = _abi.RmAreaLights()
    al.n_lights = len(radii) if n is None else n
    al.radius = None if null_radius else C.cast(a, C.POINTER(C.c_double))
    al.samples = samples
    return al


@pytest.mark.parametrize("kw", [None, dict(samples=0), dict(samples=9), dict(radii=(0., -1.)), dict(radii=(np.nan, 1.)),
                                dict(radii=(np.inf, 1.)), dict(null_radius=True), dict(n=-1)])
def test_invalid_lights_are_rejected_without_a_device(kw):
    assert _call(lights=None if kw is None else _lights(**kw)) == INVALID


def test_invalid_parameters_are_rejected_without_a_device():
    L = _abi.load()
    assert _call(lights=_lights(), rgb=False) == INVALID
    for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
        p = _abi.RmParams()
        L.rm_params_default(C.byref(p), 64, 64)
        setattr(p, field, value)
        assert _call(params=p, lights=_lights()) == INVALID, field


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    assert _call(lights=_lights()) == NOT_INITIALISED
    assert _call(lights=_lights(samples=1)) == NOT_INITIALISED     # (rm_render's frame)


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(samples=True), dict(radii=-1.),
                                dict(radii=np.nan), dict(radii=(1., 2., 3.)), dict(radii=(1., np.inf)), dict(patch_rows=(0, -1, 2))])
def test_renderer_rejects_invalid_area_light_arguments(kw):
    import rusty_marcher_b200 as rm
    args = dict(radii=1.)
    args.update(kw)
    scene = rm.Scene.create_default()
    assert len(scene.lights) == 2
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_area_lights(rm.create_frame_buffer(64, 64), scene, **args)
