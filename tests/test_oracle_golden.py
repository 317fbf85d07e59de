"""Pins the oracle: golden image of the reference (engine/out.ppm), the reference's own unit tests
restated (SURVEY.md 4), and the independently derived known answers of SURVEY.md 8c."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OUT_PPM_SHA = "82d51afaaf4a644547728dde89478e484c245d2e3eb1e40da8b928ebd7584797"   # engine/out.ppm


@pytest.fixture(scope="module")
def demo_800():
    return O.render(O.Scene.create_default(), 800, 600)


def demo_ppm(r):
    rgb = r["rgb"].copy()
    O.normalize(rgb)
    return O.ppm_bytes(rgb)


def test_demo_matches_reference_golden_ppm(demo_800):
    """Byte-for-byte against the reference's golden render (800x600, fov 1.5, camera origin)."""
    ppm = demo_ppm(demo_800)
    meta = json.load(open(os.path.join(GOLDEN, "out_ppm.json")))
    assert meta["sha256"] == OUT_PPM_SHA
    assert len(ppm) == meta["size"]
    assert ppm[:15].decode("latin1") == meta["header"]
    assert [ppm[i] for i in range(0, len(ppm), meta["sample_stride"])] == meta["sample"]
    assert hashlib.sha256(ppm).hexdigest() == OUT_PPM_SHA


def test_demo_matches_reference_file_if_present(demo_800):
    """Byte-for-byte against a stored copy of the reference's engine/out.ppm (make_reference_inputs.py)."""
    with gzip.open(os.path.join(GOLDEN, "out.ppm.gz"), "rb") as f:
        ref = f.read()
    assert hashlib.sha256(ref).hexdigest() == OUT_PPM_SHA
    assert demo_ppm(demo_800) == ref


def test_rows_below_last_patch_row_are_never_rendered(demo_800):
    """renderer.rs:47-55: 600 rows -> 18 patch rows -> rows 576..599 stay zero."""
    assert np.all(demo_800["rgb"][576:] == 0.)
    assert np.all(demo_800["prim_id"][576:] == -1)
    assert demo_800["rgb"][575].max() > 0.


def test_demo_known_answers(demo_800):
    """SURVEY.md 8c: counts/pixels derived by an independent f64 restatement."""
    c = demo_800["counters"]
    expect = dict(closest_segments=867233, anyhit_segments=828954, hits=414477, glass_hits=299608,
                  reflections=199379, refractions=299608, sphere_tests=6157993, plane_tests=2942296,
                  edge_tests=4290066, pixels=460800)
    for k, v in expect.items():
        assert c[k] == v, k
    # shadowed light evaluations
    assert c["light_evals"] - c["lit_lights"] == 230836
    rgb = demo_800["rgb"]
    assert rgb.max() == 2.3621674603868565
    assert np.unravel_index(np.argmax(rgb), rgb.shape) == (278, 312, 0)
    assert rgb.mean() == 0.3441024638099151
    px = {(400, 300): (0.41865511882860496, 0.4639826782429074, 0.48371263064489023),
          (100, 100): (1.3274771956754563, 1.0417111629741056, 1.0417111629741056),
          (700, 300): (0.8773522255638875, 0.10000000000000228, 0.7801441875112234),
          (400, 500): (0.34754375164567697, 0.264, 0.28244033313614864),
          (799, 575): (0.5211352724285305, 0.9098267159874808, 0.9098267159874808)}
    for (x, y), v in px.items():
        assert tuple(rgb[y, x]) == v
    stored = json.load(open(os.path.join(GOLDEN, "oracle_demo_800x600.json")))
    assert stored["counters"] == c


def test_demo_config1_known_answers():
    """Config 1 (1600x1280): SURVEY.md 8c."""
    r = O.render(O.Scene.create_default(), 1600, 1280, want_fragile=False)
    assert r["counters"]["closest_segments"] == 3996664
    assert r["counters"]["anyhit_segments"] == 3883330
    assert r["rgb"].max() == 2.384412303490435
    assert np.unravel_index(np.argmax(r["rgb"]), r["rgb"].shape) == (593, 614, 0)
    assert hashlib.sha256(demo_ppm(r)).hexdigest() == "b0af8771541478f91f58e4f51374078fd51d974d574386a6929524b6180aa5a8"


def test_width_must_be_multiple_of_32():
    with pytest.raises(ValueError):
        O.render(O.Scene.create_default(), 100, 64)


def test_threads_and_patch_ranges_do_not_change_the_result(demo_800):
    sc = O.Scene.create_default()
    one = O.render(sc, 800, 600, threads=1, want_fragile=False, want_counters=False)
    assert np.array_equal(one["rgb"], demo_800["rgb"])
    parts = np.zeros_like(one["rgb"])
    for rows in ((0, 5), (5, 11), (11, 18)):
        O.render(sc, 800, 600, patch_rows=rows, out=parts, want_ids=False, want_fragile=False, want_counters=False)
    assert np.array_equal(parts, demo_800["rgb"])


# ---- the reference's own unit tests, restated against the oracle -------------------------------

def _v(*a):
    return (np.array(a, dtype=np.float64))


def _call3(fn, *args):
    import ctypes as C
    out = (C.c_double * 3)()
    fn(*[O._d3(a) if not np.isscalar(a) else a for a in args], out)
    return tuple(out)


def test_geometry_scale_dot_norm_cross():
    """engine/src/geometry.rs:188-408"""
    L = O.lib()
    assert _call3(L.orc_vec_scaled, (1., 1., 1.), 1.36) == (1.36, 1.36, 1.36)
    assert _call3(L.orc_vec_scaled, (1., 2., 3.), 1.36) == (1.36, 2.72, 4.08)
    assert L.orc_vec_dot(O._d3((0, 1, 0)), O._d3((1, 0, 0))) == 0.
    assert L.orc_vec_dot(O._d3((0, 1, 0)), O._d3((0, 1, 0))) == 1.
    assert L.orc_vec_dot(O._d3((0, 1, 0)), O._d3((0, -1, 0))) == -1.
    assert L.orc_vec_dot(O._d3((1, 1, 0)), O._d3((1, -1, 0))) == 0.
    assert L.orc_vec_dot(O._d3((42, 1, 0)), O._d3((42, 1, 0))) == 42. * 42. + 1.
    n = _call3(L.orc_vec_normalized, (42., 1., 0.))
    assert L.orc_vec_dot(O._d3(n), O._d3(n)) == 1.            # geometry.rs:288: exact
    assert _call3(L.orc_vec_normalized_l0, (42., 1., 0.))[0] == 1.
    assert _call3(L.orc_vec_cross, (1., 0., 0.), (0., 1., 0.)) == (0., 0., 1.)
    assert _call3(L.orc_vec_cross, (0., 1., 0.), (0., 0., 1.)) == (1., 0., 0.)


def test_optics_reflection():
    """engine/src/optics.rs:96-132"""
    import ctypes as C
    L = O.lib()
    incident, normal = (0.5, -0.5, 0.), (0., 1., 0.)
    assert _call3(L.orc_reflect, incident, normal) == (0.5, 0.5, 0.)
    ro, rd = (C.c_double * 3)(), (C.c_double * 3)()
    assert L.orc_reflect_ray(O._d3(incident), O._d3((0, 0, 0)), O._d3(normal), 1.5, ro, rd) == 1
    assert tuple(rd) == (0.5, 0.5, 0.)


def test_triangle_intersect_cyclic_orders():
    """engine/src/triangle.rs:89-138"""
    import ctypes as C
    L = O.lib()
    v = [(-1., 3., 2.2), (-3., 0.2, 2.1), (0., 1., 2.)]
    orig = (-1., 2., 5.3)
    d = _call3(L.orc_vec_normalized, (0.1, -0.2, -3.))
    res = []
    for order in ((0, 1, 2), (1, 2, 0), (2, 0, 1)):
        verts = (C.c_double * 9)(*[c for i in order for c in v[i]])
        p, n = (C.c_double * 3)(), (C.c_double * 3)()
        assert L.orc_triangle_intersect(verts, O._d3(orig), O._d3(d), p, n) == 1
        res.append((np.array(tuple(p)), np.array(tuple(n))))
    for p, n in res[1:]:
        assert ((res[0][0] - p) ** 2).sum() < 1e-3
        assert ((res[0][1] - n) ** 2).sum() < 1e-3
    assert abs((res[0][1] ** 2).sum() - 1.) < 1e-3
    assert float(res[0][1] @ np.array(d)) < 0.


# ---- OBJ ingest (tobj restatement; parity unpinned, see oracle/rm_oracle.h) ---------------------

def test_cornell_box_loads_like_the_reference_expects():
    """obj.rs:229-233 (is_some) + SURVEY.md 8c known answers, on the stored geometry of test_data/cornell_box.obj."""
    s = O.Scene()
    assert s.add_obj_file(os.path.join(GOLDEN, "cornell_box.obj")) == 8
    assert [s.obj_triangles(i).shape[0] for i in range(8)] == [6, 2, 2, 2, 2, 2, 10, 10]
    s.add_default_lights()
    r = O.render(s, 320, 256)
    hit = r["prim_id"] >= 0
    assert hit.sum() == 9402
    assert r["prim_id"][hit].min() >= 16 and r["prim_id"][hit].max() < 26      # only shape 6, short_block (prims 16..25)
    assert r["rgb"].max() == 2.9418694361863578
    assert r["degenerate_hits"] == 0


def test_dodecahedron_known_answers():
    s = O.Scene()
    assert s.add_obj_file(os.path.join(GOLDEN, "dodecahedron.obj")) == 1
    tris = s.obj_triangles(0)
    assert tris.shape[0] == 36
    s.add_default_lights()
    r = O.render(s, 320, 256)
    assert (r["prim_id"] >= 0).sum() == 2028
    assert r["rgb"].max() == 1.2948687004360002


def test_fixture_meshes_equal_the_reference_files():
    """The committed scenes/*.npz are exactly what the OBJ reader produces from the stored geometry of the reference files."""
    from rusty_marcher_b200 import workloads
    for name in ("cornell_box", "dodecahedron"):
        s = O.Scene()
        s.add_obj_file(os.path.join(GOLDEN, name + ".obj"), offset=(0., 0., 0.))
        models = workloads.load_models(name)
        assert s.num_shapes == len(models)
        for i, (_n, v) in enumerate(models):
            assert np.array_equal(s.obj_triangles(i), v)


def test_missing_obj_is_reported():
    with pytest.raises(IOError):
        O.Scene().add_obj_file("/nonexistent/file.obj")
