"""Renderer (engine/src/renderer.rs:17-135): the drop-in for the reference's render driver.

`Renderer.render(frame, scene)` keeps the reference's signature and return value (the status
string of renderer.rs:116-121) but runs the hot path on the GPU through the C ABI (rm_render)."""
import ctypes as C
import time
import types

import numpy as np

from . import _abi
from .geometry import Vec3f
from .obj import Obj


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

    def render_view(self, frame, scene, forward, up=(0., 1., 0.), prim_id=None, rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): render() from the camera turned to look along `forward`, with `up`
        (only its component orthogonal to forward matters) towards the top of the frame -- rm_render_view, or
        rm_render_view_f64 with precision RM_FP64.  The basis is view_basis(forward, up); forward = (0, 0, -1) with up =
        (0, 1, 0) is render()'s camera and frame.  Honours precision and accel like render(); fills frame.buffer (float32,
        float64 for RM_FP64) over the rendered rows and the optional prim_id / rgb8 arrays, and returns the same kind of
        status message.  Raises ValueError for an invalid view (see view_basis)."""
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        for name, a, dtype, shape in (("prim_id", prim_id, np.int32, (frame.height, frame.width)),
                                      ("rgb8", rgb8, np.uint8, (frame.height, frame.width, 3))):
            if a is not None and (not isinstance(a, np.ndarray) or a.dtype != dtype or a.shape != shape or not a.flags.c_contiguous
                                  or not a.flags.writeable):
                raise ValueError("%s must be a writeable C-contiguous %s array of shape %s" % (name, np.dtype(dtype).name, shape))
        view = _view(forward, up)
        view_basis(forward, up)                                 # ValueError for an invalid view, before any GPU work
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        p = self.params(frame, scene, patch_rows)
        want64 = self.precision == _abi.RM_FP64
        want_dtype = np.float64 if want64 else np.float32
        if frame.buffer.dtype != want_dtype or not frame.buffer.flags.c_contiguous:
            frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=want_dtype)
        stats = _abi.RmStats()
        fn = L.rm_render_view_f64 if want64 else L.rm_render_view
        _abi.check(fn(scene.device_handle(), C.byref(p), C.byref(view), frame.buffer.ctypes.data,
                      prim_id.ctypes.data if prim_id is not None else None,
                      rgb8.ctypes.data if rgb8 is not None else None, C.byref(stats)))
        self.last_stats = stats
        ms = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms if ms > 0 else float("inf")
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (ms, int(min(fps, 2**32 - 1)), fps * frame.height * frame.width / 1e6)
        print(message)
        return message

    def render_lens(self, frame, scene, aperture, focus, samples=4, forward=None, up=(0., 1., 0.), rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): depth of field.  A thin-lens camera of radius `aperture` (scene units,
        >= 0) focused at distance `focus` (> 0, along the view axis) traces samples x samples rays per pixel from points of
        the lens through the plane in focus, and the pixel is their mean (rm_render_lens).  forward / up turn the camera as
        render_view() does (forward=None: the reference's camera looking down -z).  aperture = 0 without a view is
        render_supersampled()'s frame.  Fills frame.buffer (float32) over the rendered rows and, if given, rgb8 (H, W, 3)
        uint8 with normalize + to_vec of that frame; returns the same kind of status message as render()."""
        return self._render_sampled("render_lens", frame, scene, samples, patch_rows, rgb8, lens=(aperture, focus), view=(forward, up),
                                    check_stride=False,
                                    call=lambda L, a: L.rm_render_lens(a.scene, a.params, a.view, a.lens, a.rgb, a.rgb8, a.stats))

    def render_area_lights(self, frame, scene, radii, samples=4, prim_id=None, rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): soft shadows.  Each of the scene's lights gets a radius for this frame
        (`radii`: one number for every light, or one per light in the scene's order; finite, >= 0, 0 = the reference's point
        light), and a light of radius r > 0 is sampled at samples x samples points of the disc of radius r that faces the
        shading point, each with 1 / samples^2 of its colour (rm_render_area_lights).  samples = 1, or every radius 0, is
        render()'s frame.  Fills frame.buffer (float32) over the rendered rows and, if given, prim_id (H, W) int32 (render()'s
        primary ids) and rgb8 (H, W, 3) uint8 with normalize + to_vec of that frame; returns the same kind of status message
        as render()."""
        return self._render_sampled("render_area_lights", frame, scene, samples, patch_rows, rgb8, prim_id=prim_id,
                                    effects=dict(light_radii=radii),
                                    call=lambda L, a: L.rm_render_area_lights(a.scene, a.params, a.lights, a.rgb, a.prim_id, a.rgb8, a.stats))

    def render_rough_glass(self, frame, scene, roughness, samples=4, forward=None, up=(0., 1., 0.), aperture=0., focus=1., rgb8=None,
                           patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): rough (frosted) glass.  Each shape gets a roughness g for this frame
        (`roughness`: one number for every shape, or one per entry of scene.shapes, an Obj's value covering all its triangles;
        finite, >= 0, 0 = the reference's ideal optics), and every ray a glass-like hit spawns is turned within atan(g) of its
        ideal direction, a different way for each of the samples x samples rays of a pixel; the pixel is their mean
        (rm_render_rough_glass).  forward / up turn the camera as render_view() does, aperture / focus add render_lens()'s
        thin lens (aperture 0: the pinhole).  samples = 1, or no rough glass-like shape, is render_lens()'s frame.  Fills
        frame.buffer (float32) over the rendered rows and, if given, rgb8 (H, W, 3) uint8 with normalize + to_vec of that
        frame; returns the same kind of status message as render()."""
        return self._render_sampled("render_rough_glass", frame, scene, samples, patch_rows, rgb8, effects=dict(roughness=roughness),
                                    lens=(aperture, focus), view=(forward, up),
                                    call=lambda L, a: L.rm_render_rough_glass(a.scene, a.params, a.view, a.lens, a.rough, a.rgb, a.rgb8, a.stats))

    def render_motion(self, frame, scene, displacement, samples=4, forward=None, up=(0., 1., 0.), aperture=0., focus=1., rgb8=None,
                      patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): motion blur.  Each shape moves by a displacement over the shutter
        (`displacement`: one 3-vector for every shape, or one per entry of scene.shapes, an Obj's value covering all its
        triangles; finite), the scene as given being its pose at mid-shutter; the samples x samples rays of a pixel see the
        scene at as many different times, and the pixel is their mean (rm_render_motion).  forward / up turn the camera as
        render_view() does, aperture / focus add render_lens()'s thin lens (aperture 0: the pinhole).  samples = 1, or no
        displacement at all, is render_lens()'s frame.  Fills frame.buffer (float32) over the rendered rows and, if given,
        rgb8 (H, W, 3) uint8 with normalize + to_vec of that frame; returns the same kind of status message as render()."""
        return self._render_sampled("render_motion", frame, scene, samples, patch_rows, rgb8, effects=dict(displacement=displacement),
                                    lens=(aperture, focus), view=(forward, up),
                                    call=lambda L, a: L.rm_render_motion(a.scene, a.params, a.view, a.lens, a.motion, a.rgb, a.rgb8, a.stats))

    def render_distributed(self, frame, scene, samples=4, forward=None, up=(0., 1., 0.), aperture=0., focus=1., light_radii=None,
                           roughness=None, displacement=None, rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): distributed ray tracing.  Depth of field (forward / up, aperture / focus
        as render_lens() takes them), soft shadows (light_radii as render_area_lights() takes its radii), rough glass
        (roughness as render_rough_glass() takes it) and motion blur (displacement as render_motion() takes it) in one frame:
        every one of the samples x samples rays of a pixel samples the lens, the time, one point of each area light and the
        turn of every ray rough glass spawns, and the pixel is their mean (rm_render_distributed).  None leaves an effect out.
        An area light here is one point per sample ray with the light's full colour -- not render_area_lights()'s frame.
        samples = 1, or no active effect, is render_lens()'s frame; rough glass alone is render_rough_glass()'s and motion
        alone render_motion()'s.  Fills frame.buffer (float32) over the rendered rows and, if given, rgb8 (H, W, 3) uint8 with
        normalize + to_vec of that frame; returns the same kind of status message as render()."""
        return self._render_sampled("render_distributed", frame, scene, samples, patch_rows, rgb8,
                                    effects=_given(light_radii=light_radii, roughness=roughness, displacement=displacement),
                                    lens=(aperture, focus), view=(forward, up),
                                    call=lambda L, a: L.rm_render_distributed(a.scene, a.params, a.samples, a.view, a.lens, a.lights, a.rough,
                                                                              a.motion, a.rgb, a.rgb8, a.stats))

    def render_indirect(self, frame, scene, samples=4, forward=None, up=(0., 1., 0.), aperture=0., focus=1., rgb8=None,
                        patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): diffuse interreflection.  Every opaque hit whose material has diffusion > 0
        and a non-black diffuse_color spawns one cosine-weighted diffuse ray, a different one for each of the samples x samples
        rays of a pixel, and adds what it sees weighted by diffusion * diffuse_color: colour bleeds between surfaces and
        corners darken (rm_render_indirect).  The scene's max_depth caps the whole path, bounces included.  forward / up turn
        the camera as render_view() does, aperture / focus add render_lens()'s thin lens (aperture 0: the pinhole).
        max_depth = 1, or a scene in which nothing bounces, is render_lens()'s frame.  Fills frame.buffer (float32) over the
        rendered rows and, if given, rgb8 (H, W, 3) uint8 with normalize + to_vec of that frame; returns the same kind of
        status message as render()."""
        return self._render_sampled("render_indirect", frame, scene, samples, patch_rows, rgb8, lens=(aperture, focus), view=(forward, up),
                                    call=lambda L, a: L.rm_render_indirect(a.scene, a.params, a.view, a.lens, a.samples, a.rgb, a.rgb8, a.stats))

    def render_path(self, frame, scene, samples=4, forward=None, up=(0., 1., 0.), aperture=0., focus=1., light_radii=None,
                    roughness=None, displacement=None, rgb8=None, patch_rows=(0, -1)):
        """EXTENSION MODE (no reference counterpart): path-traced frames.  render_indirect()'s diffuse bounce together with
        render_distributed()'s depth of field (forward / up, aperture / focus), soft shadows (light_radii), rough glass
        (roughness) and motion blur (displacement), each taken as render_distributed() takes it and None leaving it out: every
        one of the samples x samples rays of a pixel samples the lens, the time, one point of each area light, the turn of every
        ray rough glass spawns and the direction of every diffuse ray, and the pixel is their mean (rm_render_path).  The
        scene's max_depth caps the whole path, bounces included.  max_depth = 1, or a scene in which nothing bounces, is
        render_distributed()'s frame; otherwise samples = 1, or no active effect, is render_indirect()'s.  Fills frame.buffer
        (float32) over the rendered rows and, if given, rgb8 (H, W, 3) uint8 with normalize + to_vec of that frame; returns the
        same kind of status message as render()."""
        return self._render_sampled("render_path", frame, scene, samples, patch_rows, rgb8,
                                    effects=_given(light_radii=light_radii, roughness=roughness, displacement=displacement),
                                    lens=(aperture, focus), view=(forward, up),
                                    call=lambda L, a: L.rm_render_path(a.scene, a.params, a.samples, a.view, a.lens, a.lights, a.rough, a.motion,
                                                                       a.rgb, a.rgb8, a.stats))

    def _render_sampled(self, name, frame, scene, samples, patch_rows, rgb8, call, prim_id=None, effects=None, lens=None, view=None,
                        check_stride=True):
        """The sampled-frame methods: validates their arguments in one order -- samples, the per-light and per-primitive
        values, the lens, precision, frame size, patch-row stride, output arrays, view -- builds the C structs and makes the
        C call, call(lib, args), with args.scene, params, samples, view, lens, lights, rough, motion, rgb, prim_id, rgb8 and
        stats as the C function takes them (None: not given).  `effects` holds the effect arguments the call was given, by
        keyword (light_radii, roughness, displacement), each checked whatever its value; `lens` is (aperture, focus), `view`
        (forward, up) with forward None for the reference's camera; check_stride=False leaves the patch-row stride to the C call."""
        if not isinstance(samples, (int, np.integer)) or isinstance(samples, bool) or not 1 <= samples <= 8:
            raise ValueError("samples must be an integer in [1, 8], got %r" % (samples,))
        s = int(samples)
        effects = effects or {}
        radii = _light_radii(scene, effects["light_radii"]) if "light_radii" in effects else None
        rough_by_prim = _roughness_by_prim(scene, effects["roughness"]) if "roughness" in effects else None
        disp_by_prim = _displacement_by_prim(scene, effects["displacement"]) if "displacement" in effects else None
        if lens is not None:
            lens = _lens_values(*lens)
        if self.precision != _abi.RM_FP32:
            raise ValueError("%s computes in RM_FP32" % name)
        if int(self.width) != frame.width or int(self.height) != frame.height:
            raise ValueError("renderer was created for %dx%d, the frame is %dx%d" % (int(self.width), int(self.height), frame.width, frame.height))
        if check_stride and len(patch_rows) > 2 and patch_rows[2] > 1:
            raise ValueError("%s renders contiguous patch rows (stride <= 1)" % name)
        for what, a, dtype, shape in (("prim_id", prim_id, np.int32, (frame.height, frame.width)),
                                      ("rgb8", rgb8, np.uint8, (frame.height, frame.width, 3))):
            if a is not None and (not isinstance(a, np.ndarray) or a.dtype != dtype or a.shape != shape or not a.flags.c_contiguous
                                  or not a.flags.writeable):
                raise ValueError("%s must be a writeable C-contiguous %s array of shape %s" % (what, np.dtype(dtype).name, shape))
        a = types.SimpleNamespace(samples=s, view=None, lens=None, lights=None, rough=None, motion=None)
        if view is not None and view[0] is not None:
            a.view = C.byref(_view(*view))
            view_basis(*view)                                   # ValueError for an invalid view, before any GPU work
        if lens is not None:
            a.lens = C.byref(_abi.RmLens(lens[0], lens[1], s))
        if radii is not None:
            a.lights = C.byref(_abi.RmAreaLights(radii.shape[0], radii.ctypes.data_as(C.POINTER(C.c_double)), s))
        if rough_by_prim is not None:
            a.rough = C.byref(_abi.RmRoughGlass(rough_by_prim.shape[0], rough_by_prim.ctypes.data_as(C.POINTER(C.c_double)), s))
        if disp_by_prim is not None:
            a.motion = C.byref(_abi.RmMotion(disp_by_prim.shape[0], disp_by_prim.ctypes.data_as(C.POINTER(C.c_double)), s))
        L = _abi.load()
        _abi.init(_abi._initialised_device if _abi._initialised_device is not None else 0)
        now = time.perf_counter()
        p = self.params(frame, scene, patch_rows)
        if frame.buffer.dtype != np.float32 or not frame.buffer.flags.c_contiguous:
            frame.buffer = np.zeros((frame.height, frame.width, 3), dtype=np.float32)
        stats = _abi.RmStats()
        a.scene, a.params, a.stats = scene.device_handle(), C.byref(p), C.byref(stats)
        a.rgb, a.prim_id = frame.buffer.ctypes.data, prim_id.ctypes.data if prim_id is not None else None
        a.rgb8 = rgb8.ctypes.data if rgb8 is not None else None
        _abi.check(call(L, a))
        self.last_stats = stats
        ms = int((time.perf_counter() - now) * 1000)
        fps = 1000. / ms if ms > 0 else float("inf")
        message = "Scene rendered in %d ms (%d fps, %.2f MP/s)" % (ms, int(min(fps, 2**32 - 1)), fps * frame.height * frame.width / 1e6)
        print(message)
        return message

def _given(**effects):
    """render_distributed / render_path: the effect arguments that are not None (None leaves an effect out)."""
    return {k: v for k, v in effects.items() if v is not None}


def _light_radii(scene, radii):
    """One radius per light of the scene (one number for every light, or one per light), float64, checked."""
    n = len(scene.lights)
    r = np.asarray(radii, dtype=np.float64)
    if r.ndim == 0:
        r = np.full(n, float(r))
    if r.shape != (n,):
        raise ValueError("radii must be one number or %d (one per light of the scene), got shape %s" % (n, r.shape))
    if not (np.all(np.isfinite(r)) and np.all(r >= 0.)):
        raise ValueError("every radius must be finite and >= 0, got %r" % (r.tolist(),))
    return np.ascontiguousarray(r)


def _per_prim(scene, per_shape):
    # primitive ids: shapes in scene order, an Obj once per triangle
    return np.ascontiguousarray(np.repeat(per_shape, [s.triangles.shape[0] if isinstance(s, Obj) else 1 for s in scene.shapes], axis=0))


def _roughness_by_prim(scene, roughness):
    """The roughness of every primitive id (one number for every shape, or one per shape), float64, checked."""
    n = len(scene.shapes)
    g = np.asarray(roughness, dtype=np.float64)
    if g.ndim == 0:
        g = np.full(n, float(g))
    if g.shape != (n,):
        raise ValueError("roughness must be one number or %d (one per shape of the scene), got shape %s" % (n, g.shape))
    if not (np.all(np.isfinite(g)) and np.all(g >= 0.)):
        raise ValueError("every roughness must be finite and >= 0, got %r" % (g.tolist(),))
    return _per_prim(scene, g)


def _displacement_by_prim(scene, displacement):
    """The displacement of every primitive id (one 3-vector for every shape, or one per shape), (n_prims, 3) float64, checked."""
    n = len(scene.shapes)
    v = np.asarray(displacement, dtype=np.float64)
    if v.shape == (3,):
        v = np.tile(v, (n, 1))
    if v.shape != (n, 3):
        raise ValueError("displacement must be one 3-vector or %d (one per shape of the scene), got shape %s" % (n, v.shape))
    if not np.all(np.isfinite(v)):
        raise ValueError("every displacement must be finite, got %r" % (v.tolist(),))
    return _per_prim(scene, v)


def _lens_values(aperture, focus):
    aperture, focus = float(aperture), float(focus)
    if not (np.isfinite(aperture) and aperture >= 0.):
        raise ValueError("aperture must be finite and >= 0, got %r" % (aperture,))
    if not (np.isfinite(focus) and focus > 0.):
        raise ValueError("focus must be finite and > 0, got %r" % (focus,))
    return aperture, focus


def _view(forward, up):
    fwd, u = [float(x) for x in forward], [float(x) for x in up]
    if len(fwd) != 3 or len(u) != 3:
        raise ValueError("forward and up must have three components")
    v = _abi.RmView()
    v.forward[:] = fwd
    v.up[:] = u
    return v


def view_basis(forward, up=(0., 1., 0.)):
    """The camera basis of a view (rm_view_basis, include/rm_b200.h): a (3, 3) float64 array whose rows are u (right), v
    (up) and w (= -forward, normalised).  Raises ValueError for an invalid view: a component that is not finite, forward
    = 0, or up zero or parallel to forward.  Needs no GPU."""
    view = _view(forward, up)
    out = np.zeros((3, 3), dtype=np.float64)
    L = _abi.load()
    rc = L.rm_view_basis(C.byref(view), out.ctypes.data_as(C.POINTER(C.c_double)))
    if rc != _abi.RM_OK:
        raise ValueError(L.rm_last_error().decode("utf-8", "replace"))
    return out


def look_at(eye, target):
    """The `forward` of a camera at `eye` that looks at the point `target`: target - eye."""
    return tuple(float(t) - float(e) for e, t in zip(Vec3f.of(eye), Vec3f.of(target)))


def create_renderer(fov, height, width):
    return Renderer(fov, height, width)
