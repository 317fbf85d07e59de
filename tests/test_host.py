"""Host side above the C ABI: the scene builder (C++), the OBJ reader and the Python mirror of
the engine interface must produce exactly the values the reference computes (checked against the
oracle, which restates the same constructors independently)."""
import ctypes as C
import os

import numpy as np
import pytest

import rusty_marcher_b200 as rm
from oracle import oracle as O
from rusty_marcher_b200 import _abi, obj, workloads

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")     # stored geometry of test_data/*.obj


def flat_of_builder(b):
    return _abi.load().rm_builder_flatten(b).contents


def fields(st):
    """ctypes struct -> nested tuples (ignores padding bytes)."""
    out = []
    for name, _t in st._fields_:
        v = getattr(st, name)
        if isinstance(v, C.Structure):
            out.append(fields(v))
        elif isinstance(v, C.Array):
            out.append(tuple(v))
        else:
            out.append(v)
    return tuple(out)


def test_default_scene_python_mirror_equals_cpp_builder():
    L = _abi.load()
    b = L.rm_builder_create_default()
    try:
        fb = flat_of_builder(b)
        fp = rm.Scene.create_default().flatten().c
        assert (fb.n_shapes, fb.n_spheres, fb.n_polygons, fb.n_lights) == (6, 4, 2, 2) == (fp.n_shapes, fp.n_spheres, fp.n_polygons, fp.n_lights)
        assert [(fb.shapes[i].kind, fb.shapes[i].index) for i in range(6)] == [(fp.shapes[i].kind, fp.shapes[i].index) for i in range(6)]
        for i in range(4):
            assert fields(fb.spheres[i]) == fields(fp.spheres[i])
        for i in range(2):
            assert fields(fb.polygons[i]) == fields(fp.polygons[i])
            assert fields(fb.lights[i]) == fields(fp.lights[i])
        assert [fb.polygon_vertices[i] for i in range(21)] == [fp.polygon_vertices[i] for i in range(21)]
        # shape order of scene.rs:201-208 and the carried-over material fields
        blue, green, red, white = (fb.spheres[i] for i in range(4))
        assert tuple(blue.center) == (-0.5, -1.5, -5.) and blue.radius_square == 4. and blue.reflectance.is_glass_like == 1
        assert blue.reflectance.diffusion == 0.1 and blue.reflectance.reflection == 0.2 and blue.reflectance.specular_exponent == 100.
        assert green.reflectance.refractive_index == 1.5 and green.reflectance.is_glass_like == 0 and green.reflectance.specular == 0.8
        assert red.reflectance.specular_exponent == 100. and red.reflectance.refractive_index == 1.
        assert tuple(white.reflectance.diffuse_color) == (0.9, 0.9, 0.9)
        assert tuple(fb.lights[1].color) == (1., 0.5, 0.5) and fb.lights[1].intensity == 0.8
    finally:
        L.rm_builder_free(b)


def test_triangle_create_matches_oracle():
    """Triangle::create (triangle.rs:33-47): normals from the C++ builder, the numpy mirror and the oracle agree bit for bit."""
    rng = np.random.default_rng(7)
    v = rng.uniform(-600, 600, size=(200, 3, 3)).astype(np.float32).astype(np.float64)
    py = obj.triangles_from_vertices(v)
    L = _abi.load()
    b = L.rm_builder_new()
    try:
        L.rm_builder_add_mesh(b, v.ctypes.data_as(C.POINTER(C.c_double)), v.shape[0], None)
        f = flat_of_builder(b)
        cpp = np.ctypeslib.as_array(C.cast(f.triangles, C.POINTER(C.c_double)), shape=(200, 15)).copy()
    finally:
        L.rm_builder_free(b)
    assert np.array_equal(cpp, py)
    lib = O.lib()
    for t in range(0, 200, 17):
        p, n = (C.c_double * 3)(), (C.c_double * 3)()
        lib.orc_triangle_intersect((C.c_double * 9)(*v[t].ravel()), O._d3((0, 0, 0)), O._d3((0, 0, -1)), p, n)
        assert tuple(n) == tuple(py[t, 9:12])


def test_obj_offset_moves_vertices_and_centre_but_not_normal():
    v = np.array([[[0., 0., 0.], [1., 0., 0.], [0., 1., 0.]]])
    o = obj.Obj.from_vertices(v)
    before = o.triangles.copy()
    o.offset((0., 0., -500.))
    assert np.array_equal(o.triangles[:, 9:12], before[:, 9:12])
    assert np.array_equal(o.triangles[:, 12:15], before[:, 12:15] + [0., 0., -500.])
    assert np.array_equal(o.triangles[:, 2:9:3], before[:, 2:9:3] - 500.)


def test_gradient_colours():
    """obj.rs:125-138"""
    r = obj.gradient_reflectances(4)
    assert np.array_equal(r["diffuse_color"], [[1., 0., 1.], [.75, .25, 1.], [.5, .5, 1.], [.25, .75, 1.]])
    assert np.all(r["specular_exponent"] == 30.) and np.all(r["is_glass_like"] == 0) and np.all(r["reflection"] == 0.95)


OBJ_TEXT = """# comment
mtllib m.mtl
o first
usemtl a
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
v 0.5 2 0
f 1 2 3 4
f -5 -4 -3 -2 -1
usemtl b
f 1/1/1 2/2/2 3/3/3
usemtl b
f 3 4 5
o empty_object_is_dropped
o second
v 2 0 0.1
f 1 2 6
l 1 2
p 1
"""


def test_obj_reader_tobj_behaviour(tmp_path):
    (tmp_path / "m.mtl").write_text("newmtl a\nKd 1 0 0\nnewmtl b\nKd 0 1 0\n")
    path = tmp_path / "t.obj"
    path.write_text(OBJ_TEXT)
    models = obj.load(str(path))
    # quad -> 2, pentagon fan -> 3 | material change splits the model | same material does not | new object
    assert [(m.name, m.triangles.shape[0]) for m in models] == [("first", 5), ("first", 2), ("second", 1)]
    first = models[0].triangles[:, 0:9].reshape(-1, 3, 3)
    assert np.array_equal(first[0], [[0, 0, 0], [1, 0, 0], [1, 1, 0]])
    assert np.array_equal(first[1], [[0, 0, 0], [1, 1, 0], [0, 1, 0]])
    assert np.array_equal(first[4], [[0, 0, 0], [0, 1, 0], [.5, 2, 0]])
    assert np.array_equal(models[2].triangles[0, 0:9].reshape(3, 3), [[0, 0, 0], [1, 0, 0], [2, 0, np.float32(0.1)]])
    # the oracle's independent reader agrees
    s = O.Scene()
    assert s.add_obj_file(str(path), offset=(0, 0, 0)) == 3
    for i, m in enumerate(models):
        assert np.array_equal(s.obj_triangles(i), m.triangles[:, 0:9].reshape(-1, 3, 3))


def test_obj_load_missing_file_returns_none():
    assert obj.load("/nonexistent/thing.obj") is None          # obj.rs:53-56


def test_cornell_box_from_reference_file():
    models = obj.load(os.path.join(GOLDEN, "cornell_box.obj"))
    assert [(m.name, m.triangles.shape[0]) for m in models] == [
        ("floor", 6), ("light", 2), ("ceiling", 2), ("back_wall", 2), ("green_wall", 2), ("red_wall", 2),
        ("short_block", 10), ("tall_block", 10)]
    fixture = workloads.load_models("cornell_box")
    for m, (name, v) in zip(models, fixture):
        assert m.name == name and np.array_equal(m.triangles[:, 0:9].reshape(-1, 3, 3), v)


def test_scene_from_obj_equals_workload_scene():
    a = rm.Scene.from_obj(os.path.join(GOLDEN, "dodecahedron.obj")).flatten()
    b = workloads.scene("dodecahedron").flatten()
    assert a.c.n_triangles == b.c.n_triangles == 36
    assert np.array_equal(a._tris, b._tris) and np.array_equal(a._refl, b._refl)


def test_light_colour_is_linf_normalised():
    l = rm.create_light((0, 0, 0), (2., 1., 0.5), 0.3)
    assert tuple(l.color) == (1., 0.5, 0.25)


def test_scene_validation_errors():
    L = _abi.load()
    b = L.rm_builder_new()
    try:
        assert L.rm_builder_add_polygon(b, (C.c_double * 6)(0, 0, 0, 1, 0, 0), 2, None) == -5    # RM_ERR_SCENE, polygon.rs:18
        assert L.rm_builder_add_obj_file(b, b"/nonexistent.obj", None) == -3
    finally:
        L.rm_builder_free(b)


def test_stress_workload_is_deterministic_and_ccw():
    d1 = workloads.describe("stress", n_spheres=16, grid=4)
    d2 = workloads.describe("stress", n_spheres=16, grid=4)
    assert d1["spheres"] == d2["spheres"] and np.array_equal(d1["meshes"][0][1], d2["meshes"][0][1])
    assert d1["meshes"][0][1].shape == (32, 3, 3)
    t = obj.triangles_from_vertices(d1["meshes"][0][1])
    assert np.all(t[:, 11] > 0)                                # normal.z > 0: hittable under the z-only inside test
    full = workloads.describe("stress")
    assert len(full["spheres"]) == 4096 and full["meshes"][0][1].shape[0] == 100352


def test_framebuffer_normalize_to_vec_write_ppm(tmp_path):
    """framebuffer.rs:26-82 on the host mirror, against the oracle's restatement."""
    rng = np.random.default_rng(3)
    fb = rm.create_frame_buffer(32, 32, dtype=np.float64)
    fb.buffer[:] = rng.uniform(-0.2, 2.5, size=fb.buffer.shape)
    ref = fb.buffer.copy()
    O.normalize(ref)
    fb.normalize()
    assert np.array_equal(fb.buffer, ref)
    assert np.array_equal(fb.to_vec(), O.to_vec(ref))
    fb.write_ppm(str(tmp_path / "o.ppm"))
    assert (tmp_path / "o.ppm").read_bytes() == O.ppm_bytes(ref)


def test_rm_write_ppm_reproduces_the_reference_golden_file(tmp_path):
    """rm_write_ppm (the C-ABI FrameBuffer::write_ppm) on the oracle's normalised 800x600 demo frame: the file hashes to
    the reference's golden engine/out.ppm."""
    import hashlib
    import json
    from oracle import oracle as O
    from tests.oracle_scenes import build_oracle_scene
    from rusty_marcher_b200 import _abi
    r = O.render(build_oracle_scene(workloads.describe("demo")), 800, 600, want_ids=False, want_fragile=False, want_counters=False)
    rgb = r["rgb"].copy()
    O.normalize(rgb)
    rgb8 = np.ascontiguousarray(O.to_vec(rgb))
    path = str(tmp_path / "out.ppm")
    assert _abi.load().rm_write_ppm(path.encode(), 800, 600, rgb8.ctypes.data) == 0
    meta = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "out_ppm.json")))
    data = open(path, "rb").read()
    assert len(data) == meta["size"] and hashlib.sha256(data).hexdigest() == meta["sha256"]
    assert _abi.load().rm_write_ppm(None, 800, 600, rgb8.ctypes.data) == -3
    assert _abi.load().rm_write_ppm(str(tmp_path / "no" / "dir.ppm").encode(), 8, 8, rgb8.ctypes.data) == -3


def test_scene_fingerprint_and_flat_cache():
    """Scene.device_handle() re-uploads when the scene changed and re-marshals (flatten) only then: the fingerprint must
    see every kind of edit -- materials, vertices, offsets, lights -- and ignore the camera (a per-frame parameter)."""
    import rusty_marcher_b200 as rm
    s = workloads.scene("cornell_box")
    seen = {s._fp()}

    def changed():
        fp = s._fp()
        new = fp not in seen
        seen.add(fp)
        return new

    s.offset_camera((1., 2., 3.))
    assert not changed()
    s.shapes[0].offset((0., 0., 1.))
    assert changed()
    s.shapes[1].reflectances["refractive_index"][0] = 1.3
    assert changed()
    s.shapes[2].triangles[0, 0] += 1e-9
    assert changed()
    s.shapes[3].make_glass()
    assert changed()
    s.lights[0].intensity = 0.5
    assert changed()
    d = workloads.scene("demo")
    a = d._fp()
    d.shapes[0].reflectance.diffuse_color.x = 0.123
    b = d._fp()
    d.shapes[0].reflectance.refractive_index = 1.7
    assert len({a, b, d._fp()}) == 3
    big = workloads.scene("stress", n_spheres=8, grid=50)      # 5000 triangles, 600 KB: a large array
    keys = {big._fp()}
    mesh = big.shapes[-1]
    mesh.triangles[5, 2] += 0.25
    keys.add(big._fp())
    mesh.reflectances["is_glass_like"] = 1                      # an int32 field (a float sum of an f64 view sees a denormal: nothing)
    keys.add(big._fp())
    mesh.triangles[:] = mesh.triangles[::-1].copy()             # same triangles, other order: other colour gradient, other tie-breaks
    mesh.reflectances[:] = mesh.reflectances[::-1].copy()
    keys.add(big._fp())
    mesh.triangles[7, 0] += 1.                                  # a sum-preserving edit
    mesh.triangles[8, 0] -= 1.
    keys.add(big._fp())
    assert len(keys) == 5
    # flatten() always marshals afresh (callers may edit the result); device_handle() keeps one per fingerprint
    assert s.flatten() is not s.flatten()
    if not rm._abi.load().rm_init(0) == 0:                      # no GPU here: the upload fails after the marshalling
        with pytest.raises(rm.RmError):
            s.device_handle()
        first = s._flat
        assert first is not None
        with pytest.raises(rm.RmError):
            s.device_handle()
        assert s._flat is first                                 # unchanged scene: not marshalled again
        s.shapes[0].offset((0., 0., 1.))
        with pytest.raises(rm.RmError):
            s.device_handle()
        assert s._flat is not first


def test_renderer_rejects_buffers_it_would_overrun():
    """Renderer.render hands raw pointers to the C ABI: arrays of the wrong dtype / shape / layout, or a frame of another
    size than the renderer was created for (renderer.rs:25-33 vs 46-108), are refused before anything is rendered."""
    import rusty_marcher_b200 as rm
    sc = workloads.scene("demo")
    r = rm.create_renderer(1.5, 64, 96)
    fb = rm.create_frame_buffer(96, 64)
    for bad in (dict(prim_id=np.zeros((64, 96), dtype=np.int64)), dict(prim_id=np.zeros((64, 64), dtype=np.int32)),
                dict(prim_id=np.zeros((64, 192), dtype=np.int32)[:, ::2]), dict(rgb8=np.zeros((64, 96, 3), dtype=np.int8)),
                dict(rgb8=np.zeros((64, 96), dtype=np.uint8))):
        with pytest.raises(ValueError):
            r.render(fb, sc, **bad)
    with pytest.raises(ValueError):
        r.render(rm.create_frame_buffer(128, 64), sc)
    with pytest.raises(ValueError):
        r.render_dispersive(rm.create_frame_buffer(128, 64), sc)
