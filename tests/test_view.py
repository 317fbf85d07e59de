"""Camera orientation (rm_render_view, include/rm_b200.h RmView) without a GPU: the basis against its numpy and oracle
restatements, the oracle's turned camera against oracle.render, orientation sanity on the oracle, and the kernel code of
the view path compiled for the host (tests/emu/rm_view_emu.cpp) against the oracle."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi, workloads
from rusty_marcher_b200.renderer import look_at, view_basis
from tests import parity, view_ref
from tests.emu import emu, view_emu
from tests.oracle_scenes import build_oracle_scene


def _pairs():
    rng = np.random.default_rng(20261020)
    pairs = [(tuple(rng.normal(size=3) * 10. ** rng.uniform(-3, 3)), tuple(rng.normal(size=3) * 10. ** rng.uniform(-3, 3)))
             for _ in range(900)]
    axes = [tuple(float(v) for v in a) for a in np.vstack([np.eye(3), -np.eye(3)])]
    pairs += [(f, u) for f in axes for u in axes]                # axis-aligned, parallel and antiparallel included
    for k in range(40):                                          # up nearly parallel to forward, on both sides of the limit
        eps = 10. ** (-4 - 0.15 * k)
        pairs.append(((0., 0., -1.), (eps, 1e-3 * eps, 1.)))
        pairs.append(((1., 2., 3.), (1. + eps, 2., 3. - eps)))
    return pairs


PAIRS = _pairs()


def _library_basis(forward, up):
    try:
        return view_basis(forward, up)
    except ValueError:
        return None


def test_basis_matches_numpy_and_the_oracle_bit_for_bit():
    valid = 0
    for k, (f, u) in enumerate(PAIRS):
        lib, emu_b, ref, orc = _library_basis(f, u), view_emu.basis(f, u), view_ref.numpy_basis(f, u), view_ref.oracle_basis(f, u)
        assert (lib is None) == (ref is None) == (orc is None) == (emu_b is None), (f, u)
        if ref is None:
            continue
        valid += 1
        assert np.array_equal(lib, ref) and np.array_equal(orc, ref) and np.array_equal(emu_b, ref), (f, u)
        if k < 936:                                              # (not the nearly parallel pairs: cancellation in cross)
            assert np.allclose(ref @ ref.T, np.eye(3), atol=1e-12)   # orthonormal, right-handed: u x v = w
            assert np.allclose(np.cross(ref[0], ref[1]), ref[2], atol=1e-12)
    assert valid > 900


def test_identity_pair_gives_the_exact_identity():
    assert np.array_equal(view_basis((0., 0., -1.), (0., 1., 0.)), np.eye(3))
    assert np.array_equal(view_basis((0., 0., -7.5), (0., 3., 0.)), np.eye(3))


@pytest.mark.parametrize("forward,up", [((0., 0., 0.), (0., 1., 0.)), ((0., 0., -1.), (0., 0., 0.)), ((0., 1., 0.), (0., 2., 0.)),
                                        ((0., 1., 0.), (0., -1., 0.)), ((np.nan, 0., -1.), (0., 1., 0.)),
                                        ((0., 0., -1.), (np.inf, 1., 0.)), ((0., 0., -1.), (0., 1., -np.inf))])
def test_invalid_views_are_rejected(forward, up):
    with pytest.raises(ValueError):
        view_basis(forward, up)
    v = _abi.RmView()
    v.forward[:] = list(forward)
    v.up[:] = list(up)
    out = (C.c_double * 9)()
    assert _abi.load().rm_view_basis(C.byref(v), out) == -3
    assert view_ref.oracle_basis(forward, up) is None


def test_null_arguments_are_rejected():
    out = (C.c_double * 9)()
    assert _abi.load().rm_view_basis(None, out) == -3
    v = _abi.RmView()
    v.forward[:] = [0., 0., -1.]
    v.up[:] = [0., 1., 0.]
    assert _abi.load().rm_view_basis(C.byref(v), None) == -3


def test_look_at_is_target_minus_eye():
    assert look_at((1., 2., 3.), (4., 0., -1.)) == (3., -2., -4.)


def test_oracle_identity_view_equals_oracle_render():
    scene = O.Scene.create_default()
    ref = O.render(scene, 160, 128)
    for view in (None, view_ref.IDENTITY):
        got = view_ref.render(scene, 160, 128, view=view)
        assert np.array_equal(got["rgb"], ref["rgb"]) and np.array_equal(got["prim_id"], ref["prim_id"])
        assert np.array_equal(got["fragile"], ref["fragile"]) and got["counters"] == ref["counters"]


def test_sphere_on_plus_x_is_hit_at_the_centre_looking_along_plus_x():
    scene = O.Scene()
    scene.add_sphere((10., 0., 0.), 2.)
    scene.add_default_lights()
    r = view_ref.render(scene, 160, 128, view=((1., 0., 0.), (0., 1., 0.)))
    assert r["prim_id"][64, 80] == 0 and r["rgb"][64, 80].max() > 0.
    assert (view_ref.render(scene, 160, 128)["prim_id"] == -1).all()      # the reference's camera does not see it


def test_looking_down_the_floor_fills_the_frame_centre():
    """Straight down from 20 units into the demo scene (at the origin the camera stands in front of the floor's near
    edge, z = -3): the floor quad (shape 5) fills the centre of the frame."""
    scene = O.Scene.create_default()
    scene.offset_camera((0., 0., -20.))
    r = view_ref.render(scene, 160, 128, view=view_ref.DOWN)
    assert (r["prim_id"][48:80, 60:100] == 5).all()


def test_looking_away_from_the_scene_sees_nothing():
    r = view_ref.render(O.Scene.create_default(), 160, 128, view=((0., 0., 1.), (0., 1., 0.)))
    assert (r["prim_id"] == -1).all() and (r["rgb"] == 0.).all()   # a primary miss is black (renderer.rs:300-306)


# ---- the kernel code of the view path, compiled for the host, against the oracle's turned camera ----
CASES = [("demo", 256, 160, 3, {}), ("cornell_box", 160, 128, 3, {}), ("stress", 160, 128, 6, dict(n_spheres=64, grid=7)),
         ("ngons", 160, 128, 4, dict(n_spheres=12, n_polygons=40))]


@pytest.fixture(scope="module", params=CASES, ids=[c[0] for c in CASES])
def case(request):
    name, w, h, depth, kw = request.param
    desc = workloads.describe(name, **kw)
    return name, w, h, depth, workloads.build_scene(desc), build_oracle_scene(desc)


@pytest.mark.parametrize("view", list(view_ref.VIEWS), ids=list(view_ref.VIEWS))
def test_fp64_view_kernel_code_is_bit_exact(case, view):
    name, w, h, depth, scene, oscene = case
    ref = view_ref.render(oscene, w, h, view=view_ref.VIEWS[view], max_depth=depth)
    got = view_emu.render(scene, w, h, view_ref.VIEWS[view], precision="f64", max_depth=depth, cull=False)
    parity.check_exact(got, ref)
    assert got["counters"] == ref["counters"]


@pytest.mark.parametrize("view", list(view_ref.VIEWS), ids=list(view_ref.VIEWS))
def test_fp32_view_path_within_tolerance(case, view):
    name, w, h, depth, scene, oscene = case
    ref = view_ref.render(oscene, w, h, view=view_ref.VIEWS[view], max_depth=depth)
    got = view_emu.render(scene, w, h, view_ref.VIEWS[view], max_depth=depth)
    m = np.float32(got["rgb"].max())
    rgb8 = (np.float32(255) * np.clip(got["rgb"] * (np.float32(1) / m), 0, 1)).astype(np.uint8) if m > 0 else np.zeros(got["rgb"].shape, np.uint8)
    parity.check_fp32(got, ref, (h // 32) * 32, rgb8)
    # (a view that misses everything is no test of the path; out of sight are only the cornell box, all planar, at z = -500,
    # looking along +x, and everything but the demo scene's floor from the origin straight down)
    assert (got["prim_id"] >= 0).any() or (name == "cornell_box" and view == "forward+x") or (name != "demo" and view == "down")


@pytest.mark.parametrize("view", list(view_ref.VIEWS), ids=list(view_ref.VIEWS))
def test_hierarchy_and_strip_bound_change_no_pixel_under_a_view(case, view):
    """The rotated raster records keep the rectangle bounds of stage A exact (rect_max): strip bound and tile schedule on
    equal off; the hierarchy walk follows the world direction: on equals off."""
    name, w, h, depth, scene, _ = case
    v = view_ref.VIEWS[view]
    a = view_emu.render(scene, w, h, v, max_depth=depth)
    b = view_emu.render(scene, w, h, v, max_depth=depth, strip_bound=False)
    c = view_emu.render(scene, w, h, v, max_depth=depth, accel=True)
    for o in (b, c):
        assert np.array_equal(a["prim_id"], o["prim_id"]) and np.array_equal(a["rgb"], o["rgb"])


def test_identity_view_path_equals_the_fast_path():
    scene = workloads.scene("demo")
    a = emu.render(scene, 256, 160, "fast")
    b = view_emu.render(scene, 256, 160, view_ref.IDENTITY)
    assert np.array_equal(a["prim_id"], b["prim_id"]) and np.array_equal(a["rgb"], b["rgb"])
