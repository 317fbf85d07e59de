"""Adaptive anti-aliasing (rm_render_adaptive), the parts that need no GPU: the mask arithmetic the kernel runs
(rm::adaptive_mark, compiled for the host) against the numpy restatement of the definition, the definition over the oracle
and its row composition, and the argument checks of the Python mirror.  GPU part: tests/test_zz_adaptive_gpu.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from rusty_marcher_b200 import _abi
from tests import adaptive_ref as AR
from tests import supersample_ref as SS
from tests.conftest import ROOT, has_gpu

CONTRASTS = [0., 0.1, float("inf"), -1.]


@pytest.fixture(scope="module")
def mark_emu(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("emu") / "librm_adaptive_emu.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", lib,
                    os.path.join(ROOT, "tests", "emu", "rm_adaptive_emu.cpp")], check=True)
    L = C.CDLL(lib)
    L.emu_adaptive_mark.restype = C.c_int
    L.emu_adaptive_mark.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]

    def run(rgb, ids, contrast, rows=None):
        """The kernel's mask over `rows` (default [0, R)), from the 1x frame rows the kernel would see: the call's rows and
        one patch row on either side, clipped to [0, R)."""
        h, w = ids.shape
        R = 32 * (h // 32)
        r0, r1 = (0, R) if rows is None else rows
        lo, hi = max(r0 - 32, 0), min(r1 + 32, R)
        rgb = np.ascontiguousarray(rgb[lo:hi], dtype=np.float32)
        ids = np.ascontiguousarray(ids[lo:hi], dtype=np.int32)
        out = np.zeros((h, w), dtype=np.uint8)
        part = np.zeros((r1 - r0, w), dtype=np.uint8)
        assert L.emu_adaptive_mark(rgb.ctypes.data, ids.ctypes.data, w, lo, hi, r0, r1 - r0, float(np.float32(contrast)),
                                   int(contrast < 0), part.ctypes.data) == 0
        out[r0:r1] = part
        return out
    return run


def random_frame(rng, h, w):
    """Values over many binades with ties, zeros and runs of equal pixels; ids that differ only by a miss (-1)."""
    rgb = (rng.random((h, w, 3)) * np.exp2(rng.integers(-30, 8, (h, w, 3)))).astype(np.float32)
    rgb[rng.random((h, w)) < 0.15] = 0.
    flat = rng.random((h, w)) < 0.3                             # copies of the left neighbour: equal pixels
    for y, x in zip(*np.nonzero(flat)):
        if x:
            rgb[y, x] = rgb[y, x - 1]
    tie = rng.random((h, w, 3)) < 0.05                          # a channel equal to the neighbour's times 1.5: a = 3 b ...
    rgb[:, 1:][tie[:, 1:]] = (rgb[:, :-1] * np.float32(1.5))[tie[:, 1:]]
    ids = rng.integers(-1, 1, (h, w)).astype(np.int32)         # only 0 and -1 (a miss)
    ids[rng.random((h, w)) < 0.6] = 0
    return rgb, ids


@pytest.mark.parametrize("contrast", CONTRASTS)
@pytest.mark.parametrize("h", [96, 100])                       # 100: R = 96 < H, the last rows are never rendered
def test_kernel_mark_is_the_definition_on_random_frames(mark_emu, contrast, h):
    rng = np.random.default_rng(7 + h)
    rgb, ids = random_frame(rng, h, 64)
    want = AR.mark(rgb, ids, contrast)
    got = mark_emu(rgb, ids, contrast)
    assert np.array_equal(got, want)
    assert not want[96:].any() and want[:96].any()
    for rows in ((0, 32), (32, 64), (64, 96)):                 # call rows with their halo: the same mask rows
        part = mark_emu(rgb, ids, contrast, rows)
        assert np.array_equal(part[rows[0]:rows[1]], want[rows[0]:rows[1]]) and not np.delete(part, np.s_[rows[0]:rows[1]], 0).any()


def test_mask_cases_by_hand():
    z = np.zeros((32, 32, 3), dtype=np.float32)
    ids = np.zeros((32, 32), dtype=np.int32)
    assert not AR.mark(z, ids, 0.).any()                       # equal neighbours: |0 - 0| > 0 * 0 is false
    ids[5, 5] = -1                                              # one miss: itself and its 8 neighbours
    m = AR.mark(z, ids, float("inf"))
    assert m.sum() == 9 and m[4:7, 4:7].all()
    ids[:] = 0
    v = np.ones_like(z)
    v[10, 11] = [1.5, 1., 1.]                                   # |1.5 - 1| = 0.5 > k 2.5 for k < 0.2 (float32(0.2) 2.5 = 0.5)
    m = AR.mark(v, ids, 0.19)
    assert m.sum() == 9 and m[9:12, 10:13].all() and not AR.mark(v, ids, 0.2).any()
    assert not AR.mark(v, ids, float("inf")).any()
    assert AR.mark(z, ids, -1.).all() and AR.mark(z, ids, -1e-300).all()
    corner = AR.mark(z, ids, 0.)
    corner[0, 0] = 0
    assert not corner.any()


@pytest.mark.parametrize("contrast", CONTRASTS)
def test_kernel_mark_of_an_oracle_frame(mark_emu, contrast):
    r = O.render(O.Scene.create_default(), 256, 176, want_fragile=False, want_counters=False)
    rgb, ids = r["rgb"].astype(np.float32), r["prim_id"]
    want = AR.mark(rgb, ids, contrast)
    assert np.array_equal(mark_emu(rgb, ids, contrast), want)
    if contrast >= 0:
        assert 0 < want.sum() < 160 * 256


def test_definition_over_the_oracle_and_its_rows():
    scene = O.Scene.create_default()
    w, h, s = 128, 160, 2
    full = AR.render_adaptive(scene, w, h, s, 0.1)
    p = O.render(scene, w, h, want_fragile=False, want_counters=False)
    sup = SS.render_supersampled(scene, w, h, s)["rgb"]
    m = AR.mark(p["rgb"].astype(np.float32), p["prim_id"], 0.1)
    assert np.array_equal(full["mask"], m) and 0 < m.sum() < 160 * 128
    assert np.array_equal(full["rgb"], AR.compose(m, sup, p["rgb"]))
    part = AR.render_adaptive(scene, w, h, s, 0.1, patch_rows=(1, 3))
    assert np.array_equal(part["rgb"][32:96], full["rgb"][32:96]) and np.array_equal(part["mask"][32:96], full["mask"][32:96])
    assert not part["rgb"][:32].any() and not part["rgb"][96:].any() and not part["mask"][:32].any() and not part["mask"][96:].any()
    # the mask of rows 32 and 95 depends on rows 31 and 96, outside the call
    assert full["mask"][[32, 95]].any()
    assert np.array_equal(AR.render_adaptive(scene, w, h, s, -1.)["rgb"], sup)
    assert np.array_equal(AR.render_adaptive(scene, w, h, 1, 0.1)["rgb"][:160], p["rgb"][:160])


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_gpu_means_not_initialised():
    L = _abi.load()
    p = _abi.RmParams()
    L.rm_params_default(C.byref(p), 64, 64)
    out = np.zeros((64, 64, 3), dtype=np.float32)
    assert L.rm_render_adaptive(1, C.byref(p), 2, 0.1, out.ctypes.data, None, None, None) == -2      # RM_ERR_NOT_INITIALISED


@pytest.mark.parametrize("kw", [dict(samples=0), dict(samples=9), dict(samples=2.0), dict(samples=True),
                                dict(contrast=float("nan")), dict(contrast="0.1"), dict(contrast=None), dict(contrast=True),
                                dict(contrast=1j)])
def test_renderer_rejects_bad_samples_and_contrast(kw):
    import rusty_marcher_b200 as rm
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_adaptive(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), **kw)


@pytest.mark.parametrize("mask", [np.zeros((64, 64), dtype=np.int32), np.zeros((64, 32), dtype=np.uint8),
                                  np.zeros((64, 128), dtype=np.uint8)[:, ::2], "mask"])
def test_renderer_rejects_a_bad_mask(mask):
    import rusty_marcher_b200 as rm
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_adaptive(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), mask=mask)


def test_renderer_rejects_a_read_only_mask():
    import rusty_marcher_b200 as rm
    m = np.zeros((64, 64), dtype=np.uint8)
    m.flags.writeable = False
    with pytest.raises(ValueError):
        rm.create_renderer(1.5, 64, 64).render_adaptive(rm.create_frame_buffer(64, 64), rm.Scene.create_default(), mask=m)
