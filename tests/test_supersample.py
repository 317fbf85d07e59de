"""Supersampled anti-aliasing (rm_render_supersampled), the parts that need no GPU: the definition over the oracle, the
resolve arithmetic the kernel runs (rm::resolve_box, compiled for the host) against the normative order restated in numpy,
and the argument checks of the Python mirror.  GPU part: tests/test_zz_supersample_gpu.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi
from tests import supersample_ref as SS
from tests.conftest import ROOT, has_gpu


@pytest.fixture(scope="module")
def resolve_emu(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("emu") / "librm_resolve_emu.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", lib,
                    os.path.join(ROOT, "tests", "emu", "rm_resolve_emu.cpp")], check=True)
    L = C.CDLL(lib)
    L.emu_resolve_box.restype = C.c_int
    L.emu_resolve_box.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]

    def run(sub, s):
        sub = np.ascontiguousarray(sub, dtype=np.float32)
        rows, w = sub.shape[0] // s, sub.shape[1] // s
        out = np.full((rows, w, 3), np.nan, dtype=np.float32)
        assert L.emu_resolve_box(sub.ctypes.data, s, w, rows, out.ctypes.data) == 0
        return out
    return run


def test_one_sample_is_the_oracle_frame():
    a = O.render(O.Scene.create_default(), 256, 160, want_ids=False, want_fragile=False, want_counters=False)["rgb"]
    b = SS.render_supersampled(O.Scene.create_default(), 256, 160, 1)["rgb"]
    assert np.array_equal(a, b)


def test_definition_renders_only_the_sub_rows_of_the_call():
    # H = 176: floor(2 H / 32) = 11 bands of the 2x frame, but only 2 * floor(H / 32) = 10 belong to the output rows
    r = SS.render_supersampled(O.Scene.create_default(), 128, 176, 2)["rgb"]
    assert r[:160].any() and not r[160:].any()
    part = SS.render_supersampled(O.Scene.create_default(), 128, 176, 2, patch_rows=(1, 3))["rgb"]
    assert np.array_equal(part[32:96], r[32:96]) and not part[:32].any() and not part[96:].any()


@pytest.mark.parametrize("s", range(1, 9))
def test_kernel_resolve_is_the_normative_order(resolve_emu, s):
    """The resolve arithmetic of the kernel, bit for bit against numpy.  Values spread over many binades, so that the
    order of the additions shows in the last bits."""
    rng = np.random.default_rng(1000 + s)
    w, rows = 64, 5
    sub = (rng.random((s * rows, s * w, 3)) * np.exp2(rng.integers(-20, 4, (s * rows, s * w, 3)))).astype(np.float32)
    got = resolve_emu(sub, s)
    want = SS.resolve_f32(sub, s)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    if s >= 3:                                                  # a different order would give different bits somewhere
        other = np.zeros_like(want)
        for j in range(s):
            for i in range(s):
                other = other + sub[i::s, j::s]
        assert not np.array_equal(other / np.float32(s * s), want)


def test_kernel_resolve_of_a_rendered_frame(resolve_emu):
    sub = O.render(O.Scene.create_default(), 3 * 96, 3 * 64, want_ids=False, want_fragile=False, want_counters=False)["rgb"]
    sub = sub.astype(np.float32)
    assert np.array_equal(resolve_emu(sub, 3), SS.resolve_f32(sub, 3))


def test_rgb8_of_follows_the_tonemap():
    v = np.array([[[0., 0.5, 1.]], [[2., 4., 1e-9]]], dtype=np.float32)
    assert SS.rgb8_of(v, 4.).tolist() == [[[0, 31, 63]], [[127, 255, 0]]]
    assert SS.rgb8_of(np.zeros_like(v), 0.).tolist() == [[[0, 0, 0]], [[0, 0, 0]]]


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    L = _abi.load()
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    assert L.rm_render_supersampled(1, C.byref(p), 2, out.ctypes.data, None, None) == -2      # RM_ERR_NOT_INITIALISED


@pytest.mark.parametrize("samples", [0, 9, -1, 2.0, True])
def test_renderer_rejects_samples_outside_one_to_eight(samples):
    import rusty_marcher_b200 as rm
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_supersampled(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), samples)
