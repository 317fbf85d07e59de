"""The argument checks and the routing of the sampled-frame calls (rm_render_lens, rm_render_area_lights, rm_render_rough_glass,
rm_render_motion, rm_render_distributed, rm_render_indirect, rm_render_path; include/rm_b200.h) as one table: for every
rejection, the status code and the rm_last_error() text, and for the Python methods the ValueError message.  The GPU part pins
the scene-dependent rejections and one routed case per row of the routing table (rm_api.cu's route_of)."""
import ctypes as C

import numpy as np
import pytest

from rusty_marcher_b200 import _abi
from tests.conftest import has_gpu
from tests.emu import lens_emu
from tests.test_path import _struct

W = H = 64
CALLS = ("lens", "area", "rough", "motion", "distributed", "indirect", "path")
STRUCTS = {"lens": (), "area": ("lights",), "rough": ("rough",), "motion": ("motion",), "distributed": ("lights", "rough", "motion"),
           "indirect": (), "path": ("lights", "rough", "motion")}


def _bad_view():
    v = _abi.RmView()
    v.forward[:] = [0., 1., 0.]
    v.up[:] = [0., 2., 0.]
    return v


def call(name, scene=1, samples=2, params=None, view=None, lens="default", rgb=True, rgb8=False, **given):
    """One C call with valid arguments except for what is given: params fields as `params`, a struct as `lights` / `rough` /
    `motion` (None: absent), the lens as `lens` ("default": a valid lens of `samples`).  Returns (status, rm_last_error())."""
    L = _abi.load()
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), W, H)
    for k, v in (params or {}).items():
        setattr(p, k, v)
    if lens == "default":
        lens = lens_emu.lens(0.5, 10., samples)
    st = {k: given.get(k, _struct(k, n=2, samples=samples)) for k in STRUCTS[name]}
    out = np.zeros((max(p.height, 1), max(p.width, 1), 3), dtype=np.float32)
    out8 = np.zeros_like(out, dtype=np.uint8)
    ref = lambda x: C.byref(x) if x is not None else None     # noqa: E731
    o, o8 = out.ctypes.data if rgb else None, out8.ctypes.data if rgb8 else None
    if name == "lens":
        rc = L.rm_render_lens(scene, C.byref(p), ref(view), ref(lens), o, o8, None)
    elif name == "area":
        rc = L.rm_render_area_lights(scene, C.byref(p), ref(st["lights"]), o, None, o8, None)
    elif name == "rough":
        rc = L.rm_render_rough_glass(scene, C.byref(p), ref(view), ref(lens), ref(st["rough"]), o, o8, None)
    elif name == "motion":
        rc = L.rm_render_motion(scene, C.byref(p), ref(view), ref(lens), ref(st["motion"]), o, o8, None)
    elif name == "indirect":
        rc = L.rm_render_indirect(scene, C.byref(p), ref(view), ref(lens), samples, o, o8, None)
    else:
        fn = L.rm_render_distributed if name == "distributed" else L.rm_render_path
        rc = fn(scene, C.byref(p), samples, ref(view), ref(lens), ref(st["lights"]), ref(st["rough"]), ref(st["motion"]), o, o8, None)
    return rc, L.rm_last_error().decode()


def _cases():
    """(id, call, kwargs): every device-free rejection the per-call test modules provoke, plus a few with several faults at once"""
    out = []
    for name in CALLS:
        def add(tag, **kw):
            out.append(("%s-%s" % (name, tag), name, kw))
        for kind in STRUCTS[name]:
            for tag, kw in (("n-1", dict(n=-1)), ("null", dict(null=True)), ("nan", dict(value=np.nan)), ("inf", dict(value=np.inf)),
                            ("neg", dict(value=-np.inf if kind == "motion" else -1.)), ("s0", dict(samples=0)), ("s9", dict(samples=9)),
                            ("s3", dict(samples=3))):
                if name != "area" or tag != "s3":                 # (rm_render_area_lights takes its samples from the lights)
                    add("%s-%s" % (kind, tag), **{kind: _struct(kind, **kw)})
            if name in ("area", "rough", "motion"):
                add("%s-none" % kind, **{kind: None})
        if name in ("distributed", "indirect", "path"):
            for s in (0, 9, -1):
                add("samples%d" % s, samples=s)
        if name != "area":
            add("view", view=_bad_view())
            for ln in ((-0.1, 10., 2), (0.5, 0., 2), (0.5, -1., 2), (np.nan, 10., 2), (np.inf, 10., 2), (0.5, np.inf, 2), (0.5, np.nan, 2),
                       (0.5, 10., 3), (0.5, 10., 0), (0.5, 10., 9)):
                if name != "lens" or ln[2] != 3:                  # (rm_render_lens takes its samples from the lens)
                    add("lens%r" % (ln,), lens=lens_emu.lens(*ln))
            if name == "lens":
                add("lens-none", lens=None)
        add("no-outputs", rgb=False)
        for field, value in (("precision", _abi.RM_FP64), ("patch_row_stride", 2), ("max_depth", 0)):
            add(field, params={field: value})
        if name != "area":
            add("width48", params=dict(width=48))
            add("wide8x", samples=8, params=dict(width=9024))
        # several faults: the first check in the call's order wins
        add("several", params=dict(precision=_abi.RM_FP64, max_depth=0), rgb=False,
            **({"view": _bad_view()} if name != "area" else {}), **{k: _struct(k, samples=3) for k in STRUCTS[name][-1:]})
    return out


CASES = _cases()

EXPECTED = {
    'lens-view': (-3, 'view: up is zero or parallel to forward'),
    'lens-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'lens-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'lens-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'lens-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'lens-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'lens-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'lens-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'lens-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'lens-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'lens-lens-none': (-3, 'lens is null'),
    'lens-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'lens-precision': (-3, 'rm_render_lens computes in RM_FP32'),
    'lens-patch_row_stride': (-3, 'rm_render_lens renders contiguous patch rows (patch_row_stride <= 1)'),
    'lens-max_depth': (-3, 'rm_render_lens needs max_depth >= 1'),
    'lens-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'lens-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'lens-several': (-3, 'view: up is zero or parallel to forward'),
    'area-lights-n-1': (-3, 'lights: n_lights must be >= 0'),
    'area-lights-null': (-3, 'lights: radius is null'),
    'area-lights-nan': (-3, 'lights: every radius must be finite and >= 0'),
    'area-lights-inf': (-3, 'lights: every radius must be finite and >= 0'),
    'area-lights-neg': (-3, 'lights: every radius must be finite and >= 0'),
    'area-lights-s0': (-3, 'lights: samples must be in [1, 8]'),
    'area-lights-s9': (-3, 'lights: samples must be in [1, 8]'),
    'area-lights-none': (-3, 'lights is null'),
    'area-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'area-precision': (-3, 'rm_render_area_lights computes in RM_FP32'),
    'area-patch_row_stride': (-3, 'rm_render_area_lights renders contiguous patch rows (patch_row_stride <= 1)'),
    'area-max_depth': (-3, 'rm_render_area_lights needs max_depth >= 1'),
    'area-several': (-3, 'rm_render_area_lights computes in RM_FP32'),
    'rough-rough-n-1': (-3, 'rough: n_prims must be >= 0'),
    'rough-rough-null': (-3, 'rough: roughness is null'),
    'rough-rough-nan': (-3, 'rough: every roughness must be finite and >= 0'),
    'rough-rough-inf': (-3, 'rough: every roughness must be finite and >= 0'),
    'rough-rough-neg': (-3, 'rough: every roughness must be finite and >= 0'),
    'rough-rough-s0': (-3, 'rough: samples must be in [1, 8]'),
    'rough-rough-s9': (-3, 'rough: samples must be in [1, 8]'),
    'rough-rough-s3': (-3, 'rough: samples must equal lens->samples'),
    'rough-rough-none': (-3, 'rough is null'),
    'rough-view': (-3, 'view: up is zero or parallel to forward'),
    'rough-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'rough-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'rough-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'rough-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'rough-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'rough-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'rough-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'rough-lens(0.5, 10.0, 3)': (-3, 'rough: samples must equal lens->samples'),
    'rough-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'rough-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'rough-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'rough-precision': (-3, 'rm_render_rough_glass computes in RM_FP32'),
    'rough-patch_row_stride': (-3, 'rm_render_rough_glass renders contiguous patch rows (patch_row_stride <= 1)'),
    'rough-max_depth': (-3, 'rm_render_rough_glass needs max_depth >= 1'),
    'rough-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'rough-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'rough-several': (-3, 'rough: samples must equal lens->samples'),
    'motion-motion-n-1': (-3, 'motion: n_prims must be >= 0'),
    'motion-motion-null': (-3, 'motion: displacement is null'),
    'motion-motion-nan': (-3, 'motion: every displacement must be finite'),
    'motion-motion-inf': (-3, 'motion: every displacement must be finite'),
    'motion-motion-neg': (-3, 'motion: every displacement must be finite'),
    'motion-motion-s0': (-3, 'motion: samples must be in [1, 8]'),
    'motion-motion-s9': (-3, 'motion: samples must be in [1, 8]'),
    'motion-motion-s3': (-3, 'motion: samples must equal lens->samples'),
    'motion-motion-none': (-3, 'motion is null'),
    'motion-view': (-3, 'view: up is zero or parallel to forward'),
    'motion-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'motion-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'motion-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'motion-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'motion-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'motion-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'motion-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'motion-lens(0.5, 10.0, 3)': (-3, 'motion: samples must equal lens->samples'),
    'motion-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'motion-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'motion-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'motion-precision': (-3, 'rm_render_motion computes in RM_FP32'),
    'motion-patch_row_stride': (-3, 'rm_render_motion renders contiguous patch rows (patch_row_stride <= 1)'),
    'motion-max_depth': (-3, 'rm_render_motion needs max_depth >= 1'),
    'motion-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'motion-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'motion-several': (-3, 'motion: samples must equal lens->samples'),
    'distributed-lights-n-1': (-3, 'lights: n_lights must be >= 0'),
    'distributed-lights-null': (-3, 'lights: radius is null'),
    'distributed-lights-nan': (-3, 'lights: every radius must be finite and >= 0'),
    'distributed-lights-inf': (-3, 'lights: every radius must be finite and >= 0'),
    'distributed-lights-neg': (-3, 'lights: every radius must be finite and >= 0'),
    'distributed-lights-s0': (-3, 'lights: samples must be in [1, 8]'),
    'distributed-lights-s9': (-3, 'lights: samples must be in [1, 8]'),
    'distributed-lights-s3': (-3, "lights: samples must equal the call's samples"),
    'distributed-rough-n-1': (-3, 'rough: n_prims must be >= 0'),
    'distributed-rough-null': (-3, 'rough: roughness is null'),
    'distributed-rough-nan': (-3, 'rough: every roughness must be finite and >= 0'),
    'distributed-rough-inf': (-3, 'rough: every roughness must be finite and >= 0'),
    'distributed-rough-neg': (-3, 'rough: every roughness must be finite and >= 0'),
    'distributed-rough-s0': (-3, 'rough: samples must be in [1, 8]'),
    'distributed-rough-s9': (-3, 'rough: samples must be in [1, 8]'),
    'distributed-rough-s3': (-3, "rough: samples must equal the call's samples"),
    'distributed-motion-n-1': (-3, 'motion: n_prims must be >= 0'),
    'distributed-motion-null': (-3, 'motion: displacement is null'),
    'distributed-motion-nan': (-3, 'motion: every displacement must be finite'),
    'distributed-motion-inf': (-3, 'motion: every displacement must be finite'),
    'distributed-motion-neg': (-3, 'motion: every displacement must be finite'),
    'distributed-motion-s0': (-3, 'motion: samples must be in [1, 8]'),
    'distributed-motion-s9': (-3, 'motion: samples must be in [1, 8]'),
    'distributed-motion-s3': (-3, "motion: samples must equal the call's samples"),
    'distributed-samples0': (-3, 'rm_render_distributed: samples must be in [1, 8]'),
    'distributed-samples9': (-3, 'rm_render_distributed: samples must be in [1, 8]'),
    'distributed-samples-1': (-3, 'rm_render_distributed: samples must be in [1, 8]'),
    'distributed-view': (-3, 'view: up is zero or parallel to forward'),
    'distributed-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'distributed-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'distributed-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'distributed-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'distributed-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'distributed-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'distributed-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'distributed-lens(0.5, 10.0, 3)': (-3, "lens: samples must equal the call's samples"),
    'distributed-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'distributed-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'distributed-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'distributed-precision': (-3, 'rm_render_distributed computes in RM_FP32'),
    'distributed-patch_row_stride': (-3, 'rm_render_distributed renders contiguous patch rows (patch_row_stride <= 1)'),
    'distributed-max_depth': (-3, 'rm_render_distributed needs max_depth >= 1'),
    'distributed-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'distributed-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'distributed-several': (-3, "motion: samples must equal the call's samples"),
    'indirect-samples0': (-3, 'rm_render_indirect: samples must be in [1, 8]'),
    'indirect-samples9': (-3, 'rm_render_indirect: samples must be in [1, 8]'),
    'indirect-samples-1': (-3, 'rm_render_indirect: samples must be in [1, 8]'),
    'indirect-view': (-3, 'view: up is zero or parallel to forward'),
    'indirect-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'indirect-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'indirect-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'indirect-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'indirect-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'indirect-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'indirect-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'indirect-lens(0.5, 10.0, 3)': (-3, "lens: samples must equal the call's samples"),
    'indirect-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'indirect-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'indirect-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'indirect-precision': (-3, 'rm_render_indirect computes in RM_FP32'),
    'indirect-patch_row_stride': (-3, 'rm_render_indirect renders contiguous patch rows (patch_row_stride <= 1)'),
    'indirect-max_depth': (-3, 'rm_render_indirect needs max_depth >= 1'),
    'indirect-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'indirect-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'indirect-several': (-3, 'view: up is zero or parallel to forward'),
    'path-lights-n-1': (-3, 'lights: n_lights must be >= 0'),
    'path-lights-null': (-3, 'lights: radius is null'),
    'path-lights-nan': (-3, 'lights: every radius must be finite and >= 0'),
    'path-lights-inf': (-3, 'lights: every radius must be finite and >= 0'),
    'path-lights-neg': (-3, 'lights: every radius must be finite and >= 0'),
    'path-lights-s0': (-3, 'lights: samples must be in [1, 8]'),
    'path-lights-s9': (-3, 'lights: samples must be in [1, 8]'),
    'path-lights-s3': (-3, "lights: samples must equal the call's samples"),
    'path-rough-n-1': (-3, 'rough: n_prims must be >= 0'),
    'path-rough-null': (-3, 'rough: roughness is null'),
    'path-rough-nan': (-3, 'rough: every roughness must be finite and >= 0'),
    'path-rough-inf': (-3, 'rough: every roughness must be finite and >= 0'),
    'path-rough-neg': (-3, 'rough: every roughness must be finite and >= 0'),
    'path-rough-s0': (-3, 'rough: samples must be in [1, 8]'),
    'path-rough-s9': (-3, 'rough: samples must be in [1, 8]'),
    'path-rough-s3': (-3, "rough: samples must equal the call's samples"),
    'path-motion-n-1': (-3, 'motion: n_prims must be >= 0'),
    'path-motion-null': (-3, 'motion: displacement is null'),
    'path-motion-nan': (-3, 'motion: every displacement must be finite'),
    'path-motion-inf': (-3, 'motion: every displacement must be finite'),
    'path-motion-neg': (-3, 'motion: every displacement must be finite'),
    'path-motion-s0': (-3, 'motion: samples must be in [1, 8]'),
    'path-motion-s9': (-3, 'motion: samples must be in [1, 8]'),
    'path-motion-s3': (-3, "motion: samples must equal the call's samples"),
    'path-samples0': (-3, 'rm_render_path: samples must be in [1, 8]'),
    'path-samples9': (-3, 'rm_render_path: samples must be in [1, 8]'),
    'path-samples-1': (-3, 'rm_render_path: samples must be in [1, 8]'),
    'path-view': (-3, 'view: up is zero or parallel to forward'),
    'path-lens(-0.1, 10.0, 2)': (-3, 'lens: aperture must be >= 0'),
    'path-lens(0.5, 0.0, 2)': (-3, 'lens: focus must be > 0'),
    'path-lens(0.5, -1.0, 2)': (-3, 'lens: focus must be > 0'),
    'path-lens(nan, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'path-lens(inf, 10.0, 2)': (-3, 'lens: aperture and focus must be finite'),
    'path-lens(0.5, inf, 2)': (-3, 'lens: aperture and focus must be finite'),
    'path-lens(0.5, nan, 2)': (-3, 'lens: aperture and focus must be finite'),
    'path-lens(0.5, 10.0, 3)': (-3, "lens: samples must equal the call's samples"),
    'path-lens(0.5, 10.0, 0)': (-3, 'lens: samples must be in [1, 8]'),
    'path-lens(0.5, 10.0, 9)': (-3, 'lens: samples must be in [1, 8]'),
    'path-no-outputs': (-3, 'out_rgb and out_rgb8 are both null'),
    'path-precision': (-3, 'rm_render_path computes in RM_FP32'),
    'path-patch_row_stride': (-3, 'rm_render_path renders contiguous patch rows (patch_row_stride <= 1)'),
    'path-max_depth': (-3, 'rm_render_path needs max_depth >= 1'),
    'path-width48': (-4, 'Dimensions mismatch: width must be a multiple of 32 (renderer.rs:49-51,107)'),
    'path-wide8x': (-4, 'width and height must be below 65536 (and the frame below 2^22 patches)'),
    'path-several': (-3, "motion: samples must equal the call's samples"),
}


@pytest.mark.parametrize("cid,name,kw", CASES, ids=[c[0] for c in CASES])
def test_c_rejections_keep_their_status_and_message(cid, name, kw):
    assert call(name, **kw) == EXPECTED[cid]


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
@pytest.mark.parametrize("name", CALLS)
def test_valid_calls_without_a_device_are_not_initialised(name):
    want = (-2, "rm_init() has not been called (or failed): no CUDA device bound")
    assert call(name) == want
    assert call(name, lens=lens_emu.lens(0., 1., 2), **{k: None for k in STRUCTS[name] if name in ("distributed", "path")}) == want


# ---- the Python methods: the same ValueError for every input ----
def _py_cases():
    lens_kw = [dict(aperture=-1.), dict(focus=0.), dict(aperture=np.nan), dict(forward=(0., 1., 0.), up=(0., 1., 0.))]
    samples_kw = [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(samples=True)]
    stride = [dict(patch_rows=(0, -1, 2))]
    radii = [dict(light_radii=-1.), dict(light_radii=(1., 2., 3.)), dict(light_radii=(1., np.inf))]
    rough = [dict(roughness=np.nan), dict(roughness=[0.1, 0.2]), dict(roughness=-1.)]
    motion = [dict(displacement=[np.nan, 0., 0.]), dict(displacement=[0.1, 0.2])]
    outs = [dict(rgb8=np.zeros((64, 64, 3), dtype=np.float32)), dict(rgb8=np.zeros((32, 64, 3), dtype=np.uint8))]
    size = [dict(frame=(32, 64))]
    absent = [dict(light_radii=None, roughness=None, displacement=None)]       # None leaves an effect out: the C call is reached
    fp64 = [dict(precision=_abi.RM_FP64)]
    order = [dict(samples=0, aperture=-1., precision=_abi.RM_FP64), dict(aperture=-1., precision=_abi.RM_FP64, frame=(32, 64)),
             dict(precision=_abi.RM_FP64, frame=(32, 64), patch_rows=(0, -1, 2)), dict(frame=(32, 64), patch_rows=(0, -1, 2))]
    table = {
        "render_lens": (dict(aperture=0.5, focus=10.), samples_kw + lens_kw + stride + outs + size + fp64 + order[:3]),
        "render_area_lights": (dict(radii=1.), samples_kw + [dict(radii=-1.), dict(radii=(1., 2., 3.)), dict(radii=np.nan)] + stride + outs
                               + [dict(prim_id=np.zeros((64, 64), dtype=np.int64))] + size + fp64 + [dict(samples=0, radii=-1.), order[3]]
                               + [dict(radii=None), dict(samples=0, radii=None)]),
        "render_rough_glass": (dict(roughness=0.1), samples_kw + [dict(roughness=-1.), dict(roughness=[0.1, 0.2]), dict(roughness=np.inf)]
                               + lens_kw + stride + outs + size + fp64 + order + [dict(roughness=-1., aperture=-1.)]
                               + [dict(roughness=None), dict(roughness=None, aperture=-1.)]),
        "render_motion": (dict(displacement=(0.5, 0., 0.)), samples_kw + [dict(displacement=[np.nan, 0., 0.]), dict(displacement=[0.1, 0.2])]
                          + lens_kw + stride + outs + size + fp64 + order + [dict(displacement=[0.1], aperture=-1.)]
                          + [dict(displacement=None), dict(displacement=None, aperture=-1.)]),
        "render_distributed": (dict(light_radii=1., roughness=0.1, displacement=(0.5, 0., 0.)),
                               samples_kw + radii + rough + motion + lens_kw + stride + outs + size + fp64 + order
                               + [dict(light_radii=-1., roughness=-1.), dict(roughness=-1., displacement=[0.1])] + absent),
        "render_indirect": ({}, samples_kw + lens_kw + stride + outs + size + fp64 + order),
        "render_path": (dict(light_radii=1., roughness=0.1, displacement=(0.5, 0., 0.)),
                        samples_kw + radii + rough + motion + lens_kw + stride + outs + size + fp64 + order
                        + [dict(light_radii=-1., roughness=-1.), dict(roughness=-1., displacement=[0.1])] + absent),
    }
    out = []
    for method, (base, bad) in table.items():
        for k, kw in enumerate(bad):
            out.append(("%s-%d" % (method, k), method, base, kw))
    return out


PY_CASES = _py_cases()
PY_EXPECTED = {
    'render_lens-0': 'samples must be an integer in [1, 8], got 0',
    'render_lens-1': 'samples must be an integer in [1, 8], got 9',
    'render_lens-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_lens-3': 'samples must be an integer in [1, 8], got True',
    'render_lens-4': 'aperture must be finite and >= 0, got -1.0',
    'render_lens-5': 'focus must be finite and > 0, got 0.0',
    'render_lens-6': 'aperture must be finite and >= 0, got nan',
    'render_lens-7': 'view: up is zero or parallel to forward',
    'render_lens-8': 'RmError',
    'render_lens-9': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_lens-10': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_lens-11': 'renderer was created for 64x64, the frame is 64x32',
    'render_lens-12': 'render_lens computes in RM_FP32',
    'render_lens-13': 'samples must be an integer in [1, 8], got 0',
    'render_lens-14': 'aperture must be finite and >= 0, got -1.0',
    'render_lens-15': 'render_lens computes in RM_FP32',
    'render_area_lights-0': 'samples must be an integer in [1, 8], got 0',
    'render_area_lights-1': 'samples must be an integer in [1, 8], got 9',
    'render_area_lights-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_area_lights-3': 'samples must be an integer in [1, 8], got True',
    'render_area_lights-4': 'every radius must be finite and >= 0, got [-1.0, -1.0]',
    'render_area_lights-5': 'radii must be one number or 2 (one per light of the scene), got shape (3,)',
    'render_area_lights-6': 'every radius must be finite and >= 0, got [nan, nan]',
    'render_area_lights-7': 'render_area_lights renders contiguous patch rows (stride <= 1)',
    'render_area_lights-8': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_area_lights-9': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_area_lights-10': 'prim_id must be a writeable C-contiguous int32 array of shape (64, 64)',
    'render_area_lights-11': 'renderer was created for 64x64, the frame is 64x32',
    'render_area_lights-12': 'render_area_lights computes in RM_FP32',
    'render_area_lights-13': 'samples must be an integer in [1, 8], got 0',
    'render_area_lights-14': 'renderer was created for 64x64, the frame is 64x32',
    'render_rough_glass-0': 'samples must be an integer in [1, 8], got 0',
    'render_rough_glass-1': 'samples must be an integer in [1, 8], got 9',
    'render_rough_glass-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_rough_glass-3': 'samples must be an integer in [1, 8], got True',
    'render_rough_glass-4': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_rough_glass-5': 'roughness must be one number or 6 (one per shape of the scene), got shape (2,)',
    'render_rough_glass-6': 'every roughness must be finite and >= 0, got [inf, inf, inf, inf, inf, inf]',
    'render_rough_glass-7': 'aperture must be finite and >= 0, got -1.0',
    'render_rough_glass-8': 'focus must be finite and > 0, got 0.0',
    'render_rough_glass-9': 'aperture must be finite and >= 0, got nan',
    'render_rough_glass-10': 'view: up is zero or parallel to forward',
    'render_rough_glass-11': 'render_rough_glass renders contiguous patch rows (stride <= 1)',
    'render_rough_glass-12': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_rough_glass-13': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_rough_glass-14': 'renderer was created for 64x64, the frame is 64x32',
    'render_rough_glass-15': 'render_rough_glass computes in RM_FP32',
    'render_rough_glass-16': 'samples must be an integer in [1, 8], got 0',
    'render_rough_glass-17': 'aperture must be finite and >= 0, got -1.0',
    'render_rough_glass-18': 'render_rough_glass computes in RM_FP32',
    'render_rough_glass-19': 'renderer was created for 64x64, the frame is 64x32',
    'render_rough_glass-20': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_motion-0': 'samples must be an integer in [1, 8], got 0',
    'render_motion-1': 'samples must be an integer in [1, 8], got 9',
    'render_motion-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_motion-3': 'samples must be an integer in [1, 8], got True',
    'render_motion-4': 'every displacement must be finite, got [[nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0]]',
    'render_motion-5': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape (2,)',
    'render_motion-6': 'aperture must be finite and >= 0, got -1.0',
    'render_motion-7': 'focus must be finite and > 0, got 0.0',
    'render_motion-8': 'aperture must be finite and >= 0, got nan',
    'render_motion-9': 'view: up is zero or parallel to forward',
    'render_motion-10': 'render_motion renders contiguous patch rows (stride <= 1)',
    'render_motion-11': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_motion-12': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_motion-13': 'renderer was created for 64x64, the frame is 64x32',
    'render_motion-14': 'render_motion computes in RM_FP32',
    'render_motion-15': 'samples must be an integer in [1, 8], got 0',
    'render_motion-16': 'aperture must be finite and >= 0, got -1.0',
    'render_motion-17': 'render_motion computes in RM_FP32',
    'render_motion-18': 'renderer was created for 64x64, the frame is 64x32',
    'render_motion-19': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape (1,)',
    'render_distributed-0': 'samples must be an integer in [1, 8], got 0',
    'render_distributed-1': 'samples must be an integer in [1, 8], got 9',
    'render_distributed-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_distributed-3': 'samples must be an integer in [1, 8], got True',
    'render_distributed-4': 'every radius must be finite and >= 0, got [-1.0, -1.0]',
    'render_distributed-5': 'radii must be one number or 2 (one per light of the scene), got shape (3,)',
    'render_distributed-6': 'every radius must be finite and >= 0, got [1.0, inf]',
    'render_distributed-7': 'every roughness must be finite and >= 0, got [nan, nan, nan, nan, nan, nan]',
    'render_distributed-8': 'roughness must be one number or 6 (one per shape of the scene), got shape (2,)',
    'render_distributed-9': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_distributed-10': 'every displacement must be finite, got [[nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0]]',
    'render_distributed-11': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape (2,)',
    'render_distributed-12': 'aperture must be finite and >= 0, got -1.0',
    'render_distributed-13': 'focus must be finite and > 0, got 0.0',
    'render_distributed-14': 'aperture must be finite and >= 0, got nan',
    'render_distributed-15': 'view: up is zero or parallel to forward',
    'render_distributed-16': 'render_distributed renders contiguous patch rows (stride <= 1)',
    'render_distributed-17': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_distributed-18': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_distributed-19': 'renderer was created for 64x64, the frame is 64x32',
    'render_distributed-20': 'render_distributed computes in RM_FP32',
    'render_distributed-21': 'samples must be an integer in [1, 8], got 0',
    'render_distributed-22': 'aperture must be finite and >= 0, got -1.0',
    'render_distributed-23': 'render_distributed computes in RM_FP32',
    'render_distributed-24': 'renderer was created for 64x64, the frame is 64x32',
    'render_distributed-25': 'every radius must be finite and >= 0, got [-1.0, -1.0]',
    'render_distributed-26': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_indirect-0': 'samples must be an integer in [1, 8], got 0',
    'render_indirect-1': 'samples must be an integer in [1, 8], got 9',
    'render_indirect-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_indirect-3': 'samples must be an integer in [1, 8], got True',
    'render_indirect-4': 'aperture must be finite and >= 0, got -1.0',
    'render_indirect-5': 'focus must be finite and > 0, got 0.0',
    'render_indirect-6': 'aperture must be finite and >= 0, got nan',
    'render_indirect-7': 'view: up is zero or parallel to forward',
    'render_indirect-8': 'render_indirect renders contiguous patch rows (stride <= 1)',
    'render_indirect-9': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_indirect-10': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_indirect-11': 'renderer was created for 64x64, the frame is 64x32',
    'render_indirect-12': 'render_indirect computes in RM_FP32',
    'render_indirect-13': 'samples must be an integer in [1, 8], got 0',
    'render_indirect-14': 'aperture must be finite and >= 0, got -1.0',
    'render_indirect-15': 'render_indirect computes in RM_FP32',
    'render_indirect-16': 'renderer was created for 64x64, the frame is 64x32',
    'render_path-0': 'samples must be an integer in [1, 8], got 0',
    'render_path-1': 'samples must be an integer in [1, 8], got 9',
    'render_path-2': 'samples must be an integer in [1, 8], got 2.0',
    'render_path-3': 'samples must be an integer in [1, 8], got True',
    'render_path-4': 'every radius must be finite and >= 0, got [-1.0, -1.0]',
    'render_path-5': 'radii must be one number or 2 (one per light of the scene), got shape (3,)',
    'render_path-6': 'every radius must be finite and >= 0, got [1.0, inf]',
    'render_path-7': 'every roughness must be finite and >= 0, got [nan, nan, nan, nan, nan, nan]',
    'render_path-8': 'roughness must be one number or 6 (one per shape of the scene), got shape (2,)',
    'render_path-9': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_path-10': 'every displacement must be finite, got [[nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0], [nan, 0.0, 0.0]]',
    'render_path-11': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape (2,)',
    'render_path-12': 'aperture must be finite and >= 0, got -1.0',
    'render_path-13': 'focus must be finite and > 0, got 0.0',
    'render_path-14': 'aperture must be finite and >= 0, got nan',
    'render_path-15': 'view: up is zero or parallel to forward',
    'render_path-16': 'render_path renders contiguous patch rows (stride <= 1)',
    'render_path-17': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_path-18': 'rgb8 must be a writeable C-contiguous uint8 array of shape (64, 64, 3)',
    'render_path-19': 'renderer was created for 64x64, the frame is 64x32',
    'render_path-20': 'render_path computes in RM_FP32',
    'render_path-21': 'samples must be an integer in [1, 8], got 0',
    'render_path-22': 'aperture must be finite and >= 0, got -1.0',
    'render_path-23': 'render_path computes in RM_FP32',
    'render_path-24': 'renderer was created for 64x64, the frame is 64x32',
    'render_path-25': 'every radius must be finite and >= 0, got [-1.0, -1.0]',
    'render_path-26': 'every roughness must be finite and >= 0, got [-1.0, -1.0, -1.0, -1.0, -1.0, -1.0]',
    'render_area_lights-15': 'every radius must be finite and >= 0, got [nan, nan]',
    'render_area_lights-16': 'samples must be an integer in [1, 8], got 0',
    'render_rough_glass-21': 'every roughness must be finite and >= 0, got [nan, nan, nan, nan, nan, nan]',
    'render_rough_glass-22': 'every roughness must be finite and >= 0, got [nan, nan, nan, nan, nan, nan]',
    'render_motion-20': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape ()',
    'render_motion-21': 'displacement must be one 3-vector or 6 (one per shape of the scene), got shape ()',
    'render_distributed-27': 'RmError',
    'render_path-27': 'RmError',
}


def py_call(method, base, kw):
    """The method on the default scene with a 64 x 64 frame: the ValueError's message, or "RmError" where the arguments
    reach the C call (which then fails without a device, or rejects them with one)."""
    import rusty_marcher_b200 as rm
    args = dict(base)
    args.update(kw)
    h, w = args.pop("frame", (64, 64))
    r = rm.create_renderer(1.5, 64, 64)
    r.precision = args.pop("precision", _abi.RM_FP32)
    try:
        getattr(r, method)(rm.create_frame_buffer(w, h), rm.Scene.create_default(), **args)
    except ValueError as e:
        return str(e)
    except _abi.RmError:
        return "RmError"


@pytest.mark.parametrize("cid,method,base,kw", PY_CASES, ids=[c[0] for c in PY_CASES])
def test_python_rejections_keep_their_message(cid, method, base, kw):
    assert py_call(method, base, kw) == PY_EXPECTED[cid]


# ---- GPU: the rejections that need the scene ----
@pytest.mark.gpu
def test_scene_dependent_rejections_keep_their_status_and_message(rm_gpu):
    scene = rm_gpu.Scene.create_default()
    hd = scene.device_handle()
    n_l, n_p = len(scene.lights), _abi.load().rm_scene_num_prims(hd)
    unknown = (-3, "unknown scene handle")
    lights = (-3, "lights: n_lights must equal the scene's light count")
    rough = (-3, "rough: n_prims must equal the scene's primitive count")
    motion = (-3, "motion: n_prims must equal the scene's primitive count")

    def st(kind, n=None, s=2):
        return _struct(kind, n=(n_l if kind == "lights" else n_p) if n is None else n, samples=s)

    def both(name, s=2, scene=hd, **kw):
        """the call with valid structs of s samples except for those given"""
        base = {k: st(k, s=s) for k in STRUCTS[name]}
        base.update(kw)
        return call(name, scene=scene, samples=s, lens=lens_emu.lens(0.5, 10., s), **base)

    for name in CALLS:
        assert both(name, scene=987654) == unknown, name
    assert call("lens", scene=987654, lens=lens_emu.lens(0., 1., 2)) == unknown          # the pinhole
    for s in (1, 2):                                            # the counts are checked before every route
        assert both("area", s=s, lights=st("lights", n_l + 1, s)) == lights, s
        assert both("rough", s=s, rough=st("rough", n_p - 1, s)) == rough, s
        assert both("motion", s=s, motion=st("motion", n_p + 1, s)) == motion, s
        for name in ("distributed", "path"):
            assert both(name, s=s, lights=st("lights", n_l + 1, s)) == lights, (name, s)
            assert both(name, s=s, rough=st("rough", n_p + 1, s)) == rough, (name, s)
            assert both(name, s=s, motion=st("motion", 0, s)) == motion, (name, s)
            assert both(name, s=s, lights=st("lights", 0, s), rough=st("rough", 1, s), motion=st("motion", 1, s)) == lights, (name, s)
            assert both(name, s=s, rough=st("rough", 1, s), motion=st("motion", 1, s)) == rough, (name, s)


# ---- GPU: one routed case per row of the routing table, against the call the header routes it to ----
def _rows():
    from tests.test_zz_path_gpu import YAW30
    lens = dict(forward=YAW30[0], up=YAW30[1], aperture=0.5, focus=30.)
    return [
        # (row, call, its arguments, routed-to call (None: not routed), its arguments, max_depth, kernel that renders it)
        ("B+A", "render_path", dict(lens, samples=3, which="area"), None, None, 4, "path_kernel"),
        ("B", "render_path", dict(lens, samples=3), "render_indirect", dict(lens, samples=3), 4, "indirect_kernel"),
        ("A", "render_path", dict(lens, samples=3, which="area+rough"), "render_distributed", dict(lens, samples=3, which="area+rough"), 1,
         "distributed_kernel"),
        ("R+M", "render_path", dict(samples=3, which="rough+motion"), "render_distributed", dict(samples=3, which="rough+motion"), 1,
         "distributed_kernel"),
        ("R", "render_distributed", dict(lens, samples=3, which="rough"), "render_rough_glass", dict(lens, samples=3, which="rough"), 3,
         "rough_glass_kernel"),
        ("M", "render_path", dict(lens, samples=2, which="motion"), "render_motion", dict(lens, samples=2, which="motion"), 1,
         "motion_kernel"),
        ("none-lens", "render_rough_glass", dict(lens, samples=3, roughness=0.), "render_lens", dict(lens, samples=3), 3, "lens_kernel"),
        ("none-pinhole", "render_distributed", dict(samples=3, focus=7.), "render_supersampled", dict(samples=3), 3, None),
    ]


ROWS = _rows()
SAMPLED_KERNELS = ("lens_kernel", "rough_glass_kernel", "motion_kernel", "distributed_kernel", "indirect_kernel", "path_kernel")


def _render(rm, scene, method, depth, kw, kernel=None):
    """The frame, 8-bit frame, stats and names of the kernels that ran.  With `kernel`, the frame is rendered again (it is
    deterministic) until the profiler has recorded that kernel, at most three times: torch.profiler now and then misses
    one kernel record."""
    from tests.test_zz_path_gpu import effects, kernels_run, ran
    kw = dict(kw)
    kw.update(effects(scene, kw.pop("which", "")))
    r = rm.create_renderer(1.5, 192, 320)
    r.max_depth = depth
    fb = rm.create_frame_buffer(320, 192, dtype=np.float32)
    b8 = np.zeros((192, 320, 3), dtype=np.uint8)
    for _ in range(3):
        _, names = kernels_run(lambda: getattr(r, method)(fb, scene, rgb8=b8, **kw))
        if kernel is None or ran(names, kernel):
            break
    return fb.buffer, b8, r.last_stats, names


@pytest.mark.gpu
@pytest.mark.parametrize("row", ROWS, ids=[r[0] for r in ROWS])
def test_each_route_is_the_routed_calls_frame(rm_gpu, row):
    from tests.test_zz_path_gpu import ran, same, scenes
    _, method, kw, routed, routed_kw, depth, kernel = row
    scene = scenes("stress", n_spheres=256, grid=24)[0]
    got, got8, st, names = _render(rm_gpu, scene, method, depth, kw, kernel)
    assert got.any()
    if kernel is None:                                          # (a lost profiler record cannot fail this check)
        assert not any(ran(names, k) for k in SAMPLED_KERNELS), names
    else:
        assert ran(names, kernel), names
    if routed is None:                                          # the path kernel: neither the frame without the bounce nor without the effects
        assert st.kernel_launches == 2
        for other in ("render_distributed", "render_indirect"):
            want = _render(rm_gpu, scene, other, depth, dict(kw, which=kw["which"] if other == "render_distributed" else ""))[0]
            assert not same(got, want), other
        return
    want, want8, st0, _ = _render(rm_gpu, scene, routed, depth, routed_kw)
    assert same(got, want) and np.array_equal(got8, want8)
    for f in ("kernel_launches", "max_value", "resident_prims", "d2h_bytes"):
        assert getattr(st, f) == getattr(st0, f), f
