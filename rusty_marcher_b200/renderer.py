"""Renderer (engine/src/renderer.rs:17-135): the drop-in for the reference's render driver.

`Renderer.render(frame, scene)` keeps the reference's signature and return value (the status
string of renderer.rs:116-121) but runs the hot path on the GPU through the C ABI (rm_render)."""
import ctypes as C
import time

import numpy as np

from . import _abi
from .geometry import Vec3f


class Renderer:
    ACCEL_AUTO_PRIMS = 256

    def __init__(self, fov, height, width):                     # renderer.rs:25-33
        self.fov = float(fov)
        self.height = float(height)
        self.width = float(width)
        self.max_depth = 3                                      # renderer.rs:262
        self.background = 0.1                                   # renderer.rs:40-44
        self.cull_backfacing = True
        # scene queries through the bounding-volume hierarchy (RmParams.accel; the reference's unused bounding boxes,
        # shapes.rs:34-38): False = the reference's brute-force traversal, True, or "auto" = for scenes of more than
        # ACCEL_AUTO_PRIMS primitives.  The FP32 frame is bit-identical either way.
        self.accel = False
        self.precision = _abi.RM_FP32
        # re-render loops that keep one FrameBuffer (main.rs:329-351): the frame has not been touched since this renderer's
        # previous render into it, so only tiles that held something then and are black now need clearing (RM_ROWS_RETAINED)
        self.retained = False
        self.last_stats = None

    def params(self, frame, scene, patch_rows=(0, -1)):
        p = _abi.RmParams()
        _abi.load().rm_params_default(C.byref(p), frame.width, frame.height)
        p.fov = self.fov
        p.camera[:] = list(Vec3f.of(scene.camera))
        p.max_depth = self.max_depth
        p.background = self.background
        p.precision = self.precision
        p.patch_row_begin, p.patch_row_end = patch_rows[:2]     # (begin, end[, stride]) in 32-row patch rows
        p.patch_row_stride = patch_rows[2] if len(patch_rows) > 2 else 1
        p.cull_backfacing = int(self.cull_backfacing)
        accel = self.accel
        if accel == "auto":
            accel = _abi.load().rm_scene_num_prims(scene.device_handle()) > self.ACCEL_AUTO_PRIMS
        p.accel = int(bool(accel)) if self.precision == _abi.RM_FP32 else 0
        return p

    def render(self, frame, scene, prim_id=None, rgb8=None, counters=False, patch_rows=(0, -1)):
        """Renderer::render (renderer.rs:36-126).  Fills frame.buffer rows [0, floor(H/32)*32) and
        returns the reference's status message.  Optional outputs: prim_id (H, W) int32 array,
        rgb8 (H, W, 3) uint8 array (normalize + to_vec done on device)."""
        # the reference projects with the Renderer's own width / height / ratio (renderer.rs:128-135) and indexes the
        # frame with the frame's (renderer.rs:46-108); they are the same numbers in main.rs:364-371 and must be here
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        for name, a, dtype, shape in (("prim_id", prim_id, np.int32, (frame.height, frame.width)),
                                      ("rgb8", rgb8, np.uint8, (frame.height, frame.width, 3))):
            if a is not None and (not isinstance(a, np.ndarray) or a.dtype != dtype or a.shape != shape or not a.flags.c_contiguous
                                  or not a.flags.writeable):
                raise ValueError("%s must be a writeable C-contiguous %s array of shape %s" % (name, np.dtype(dtype).name, shape))
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        patch_size = 32
        if frame.height % patch_size != 0 or frame.width % patch_size != 0:
            print("Dimensions mismatch")                        # renderer.rs:49-51
        n_patches = (frame.height // patch_size) * (frame.width // patch_size)
        print("Rendering using patches of size %d, using %d patches overall" % (patch_size, n_patches))
        p = self.params(frame, scene, patch_rows)
        handle = scene.device_handle()
        stats = _abi.RmStats()
        stats.pixels = 1 if counters else 0
        want64 = self.precision == _abi.RM_FP64
        # the frame's own type decides the delivery: float64 rows are the reference's FrameBuffer (framebuffer.rs:6-10),
        # filled from the FP32 kernels through rm_render_rows_f64; float32 is the lean form
        rows_api = not want64 and prim_id is None and rgb8 is None and not counters and (
            frame.buffer.dtype == np.float64 or self.retained) and frame.buffer.flags.c_contiguous and frame.buffer.dtype in (np.float32, np.float64)
        if rows_api:
            fn = L.rm_render_rows_f64 if frame.buffer.dtype == np.float64 else L.rm_render_rows_f32
            _abi.check(fn(handle, C.byref(p), self._row_pointers(frame), _abi.RM_ROWS_RETAINED if self.retained else 0, C.byref(stats)))
        else:
            want_dtype = np.float64 if want64 else np.float32
            if frame.buffer.dtype != want_dtype or not frame.buffer.flags.c_contiguous:
                frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=want_dtype)
            fn = L.rm_render_f64 if want64 else L.rm_render
            _abi.check(fn(handle, C.byref(p), frame.buffer.ctypes.data,
                          prim_id.ctypes.data if prim_id is not None else None,
                          rgb8.ctypes.data if rgb8 is not None else None, C.byref(stats)))
        self.last_stats = stats
        ms_render_time = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms_render_time if ms_render_time > 0 else float("inf")
        pix_scale = frame.height * frame.width / 1e6
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (
            ms_render_time, int(min(fps, 2**32 - 1)), fps * pix_scale)   # renderer.rs:116-121
        print(message)
        return message


    @staticmethod
    def _row_pointers(frame):
        """frame.buffer as the reference holds it: one pointer per pixel row (Vec<Vec<Vec3f>>), cached on the frame."""
        b = frame.buffer
        key = (b.ctypes.data, b.shape, b.dtype.str)
        cached = getattr(frame, "_rows", None)
        if cached is None or cached[0] != key:
            ptrs = (C.c_void_p * frame.height)(*[b.ctypes.data + y * b.strides[0] for y in range(frame.height)])
            frame._rows = cached = (key, ptrs)
        return cached[1]

    def render_dispersive(self, frame, scene, indices=(1.50, 1.52, 1.54), prim_id=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart; BASELINE.json configs[3], SURVEY.md 8d item 4): per-channel refractive
        indices.  Three passes of the unchanged hot path -- pass c with every glass-like material of the scene at
        indices[c] -- and channel c of the frame is channel c of pass c (rm_render_dispersive).  Fills frame.buffer like
        render() and returns the same kind of status message."""
        if self.precision != _abi.RM_FP32:
            raise ValueError("render_dispersive computes in RM_FP32")
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        if prim_id is not None and (not isinstance(prim_id, np.ndarray) or prim_id.dtype != np.int32 or prim_id.shape != (frame.height, frame.width)
                                    or not prim_id.flags.c_contiguous):
            raise ValueError("prim_id must be a C-contiguous int32 array of shape (height, width)")
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        p = self.params(frame, scene, patch_rows)
        if frame.buffer.dtype != np.float32 or not frame.buffer.flags.c_contiguous:
            frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=np.float32)
        handles = (C.c_int64 * 3)()
        stats = _abi.RmStats()
        try:
            for c, n in enumerate(indices):
                flat = scene.flatten()
                flat.set_glass_index(float(n))
                h = C.c_int64(0)
                _abi.check(L.rm_scene_upload(C.byref(flat.c), C.byref(h)))
                handles[c] = h.value
            _abi.check(L.rm_render_dispersive(handles, C.byref(p), frame.buffer.ctypes.data,
                                              prim_id.ctypes.data if prim_id is not None else None, C.byref(stats)))
        finally:
            for c in range(3):
                if handles[c]:
                    L.rm_scene_free(handles[c])
        self.last_stats = stats
        ms = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms if ms > 0 else float("inf")
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (ms, int(min(fps, 2**32 - 1)), fps * frame.height * frame.width / 1e6)
        print(message)
        return message

    def render_supersampled(self, frame, scene, samples=2, rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): anti-aliasing with samples x samples primary rays per pixel.  Pixel
        (x, y) is the mean of the FP32 frame rendered at samples times the width and height over its samples x samples
        block of sub-pixels (rm_render_supersampled; samples = 1 is render()'s frame).  Fills frame.buffer (float32) over
        the rendered rows and, if given, rgb8 (H, W, 3) uint8 with normalize + to_vec of the resolved frame; returns the
        same kind of status message as render()."""
        if not isinstance(samples, (int, np.integer)) or isinstance(samples, bool) or not 1 <= samples <= 8:
            raise ValueError("samples must be an integer in [1, 8], got %r" % (samples,))
        if self.precision != _abi.RM_FP32:
            raise ValueError("render_supersampled computes in RM_FP32")
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        if rgb8 is not None and (not isinstance(rgb8, np.ndarray) or rgb8.dtype != np.uint8 or rgb8.shape != (frame.height, frame.width, 3)
                                 or not rgb8.flags.c_contiguous or not rgb8.flags.writeable):
            raise ValueError("rgb8 must be a writeable C-contiguous uint8 array of shape %s" % ((frame.height, frame.width, 3),))
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        p = self.params(frame, scene, patch_rows)
        if frame.buffer.dtype != np.float32 or not frame.buffer.flags.c_contiguous:
            frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=np.float32)
        stats = _abi.RmStats()
        _abi.check(L.rm_render_supersampled(scene.device_handle(), C.byref(p), int(samples), frame.buffer.ctypes.data,
                                            rgb8.ctypes.data if rgb8 is not None else None, C.byref(stats)))
        self.last_stats = stats
        ms = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms if ms > 0 else float("inf")
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (ms, int(min(fps, 2**32 - 1)), fps * frame.height * frame.width / 1e6)
        print(message)
        return message

    def render_adaptive(self, frame, scene, samples=4, contrast=0.1, rgb8=None, mask=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): adaptive anti-aliasing.  A pixel gets render_supersampled()'s value
        when one of its 8 neighbours in render()'s frame has another primitive id or differs in some channel by more than
        contrast * (a + b) (contrast < 0: every pixel; +inf: geometric edges only), and render()'s value otherwise
        (rm_render_adaptive).  Fills frame.buffer (float32) over the rendered rows, rgb8 (H, W, 3) uint8 with normalize +
        to_vec of that frame if given, and mask (H, W) uint8 with 1 where a pixel was refined; returns the same kind of
        status message as render()."""
        if not isinstance(samples, (int, np.integer)) or isinstance(samples, bool) or not 1 <= samples <= 8:
            raise ValueError("samples must be an integer in [1, 8], got %r" % (samples,))
        if not isinstance(contrast, (int, float, np.integer, np.floating)) or isinstance(contrast, bool) or np.isnan(contrast):
            raise ValueError("contrast must be a real number (not NaN), got %r" % (contrast,))
        if self.precision != _abi.RM_FP32:
            raise ValueError("render_adaptive computes in RM_FP32")
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        for name, a, shape in (("rgb8", rgb8, (frame.height, frame.width, 3)), ("mask", mask, (frame.height, frame.width))):
            if a is not None and (not isinstance(a, np.ndarray) or a.dtype != np.uint8 or a.shape != shape or not a.flags.c_contiguous
                                  or not a.flags.writeable):
                raise ValueError("%s must be a writeable C-contiguous uint8 array of shape %s" % (name, shape))
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        p = self.params(frame, scene, patch_rows)
        if frame.buffer.dtype != np.float32 or not frame.buffer.flags.c_contiguous:
            frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=np.float32)
        stats = _abi.RmStats()
        _abi.check(L.rm_render_adaptive(scene.device_handle(), C.byref(p), int(samples), float(contrast), frame.buffer.ctypes.data,
                                        rgb8.ctypes.data if rgb8 is not None else None,
                                        mask.ctypes.data if mask is not None else None, C.byref(stats)))
        self.last_stats = stats
        ms = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms if ms > 0 else float("inf")
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (ms, int(min(fps, 2**32 - 1)), fps * frame.height * frame.width / 1e6)
        print(message)
        return message


def create_renderer(fov, height, width):
    return Renderer(fov, height, width)
