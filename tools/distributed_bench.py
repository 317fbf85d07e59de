"""Cost of distributed ray tracing (rm_render_distributed) on one GPU, next to rm_render_lens at the same s and view.

    python tools/distributed_bench.py [--out FILE] [--calls N]

For demo (1600x1280) and stress_4k through the hierarchy (1024 spheres + 8192 triangles, 3840x2160, accel = 1; f64 ray
geometry), at s = 2 and 4, under a camera turned 10 degrees to the left (so that rm_render_lens runs lens_kernel rather than
routing to rm_render_supersampled) and without a lens:
  * rm_render_lens, and rm_render_distributed with the effect sets {area}, {area, rough}, {area, motion}, {rough, motion} and
    {area, rough, motion} -- area: every light a sphere of radius 2; rough: roughness 0.1 on every glass-like primitive;
    motion: every shape moving by a seeded displacement of length 0.5 (one direction per shape): call time (host wall time
    around the synchronous call), the call's ms_render (device time of the traced and resolved rows) and ms_total (device time
    of the whole call, copies included), medians of N calls after 2 warm-up calls;
  * in a separate pass under torch.profiler (CUDA activities): the mean time of lens_kernel / distributed_kernel.
Every listed set runs distributed_kernel (none is routed).  Outputs: float + 8-bit frame into pinned host memory
(rm_host_alloc).  The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
import argparse
import ctypes as C
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import rusty_marcher_b200 as rm  # noqa: E402
from rusty_marcher_b200 import _abi, workloads  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from motion_bench import displacement  # noqa: E402
from supersample_bench import card  # noqa: E402

# (label, description, width, height, accel)
CASES = [("demo", workloads.describe("demo"), 1600, 1280, 0),
         ("stress_4k_bvh", workloads.describe("stress", n_spheres=1024, grid=64), 3840, 2160, 1)]
SAMPLES = (2, 4)
SETS = ("area", "area+rough", "area+motion", "rough+motion", "area+rough+motion")
RADIUS, ROUGHNESS, LENGTH = 2., 0.1, 0.5
YAW = math.radians(10.)


def glass_like(scene):
    """is_glass_like by primitive id"""
    out = []
    for s in scene.shapes:
        if hasattr(s, "reflectances"):
            out.extend(bool(f) for f in s.reflectances["is_glass_like"])
        else:
            out.append(bool(s.reflectance.is_glass_like))
    return np.array(out, dtype=bool)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    rm.init(0)
    L = _abi.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say("distributed ray tracing (rm_render_distributed), one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 2 warm-up calls; outputs: float + 8-bit frame into pinned host memory" % args.calls)
    view = _abi.RmView()
    view.forward[:] = [-math.sin(YAW), 0., -math.cos(YAW)]
    view.up[:] = [0., 1., 0.]

    def timed(fn):
        st = _abi.RmStats()
        walls, ren, tot = [], [], []
        for i in range(2 + args.calls):
            t0 = time.perf_counter()
            _abi.check(fn(st))
            t1 = time.perf_counter()
            if i >= 2:
                walls.append(1e3 * (t1 - t0))
                ren.append(st.ms_render)
                tot.append(st.ms_total)
        return float(np.median(walls)), float(np.median(ren)), float(np.median(tot))

    def kernel_ms(fn, name):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                _abi.check(fn(None))
            torch.cuda.synchronize()
        ks = [e.time_range.elapsed_us() for e in prof.events() if name in e.name and e.device_type.name == "CUDA"]
        if not ks:                                              # (kernels attached to a host-side event instead)
            ks = [k.duration for e in prof.events() for k in getattr(e, "kernels", []) if name in k.name]
        if len(ks) != 3:
            raise RuntimeError("torch.profiler recorded %d %s launches, expected 3" % (len(ks), name))
        return 1e-3 * float(np.mean(ks))

    for label, desc, w, h, accel in CASES:
        scene = workloads.build_scene(desc)
        r = rm.create_renderer(1.5, h, w)
        r.accel = bool(accel)
        fb = rm.create_frame_buffer(32, 32)
        fb.width, fb.height = w, h
        p = r.params(fb, scene)
        hd = scene.device_handle()
        out = L.rm_host_alloc(h * w * 12)
        out8 = L.rm_host_alloc(h * w * 3)
        radii = np.full(len(scene.lights), RADIUS)
        g = np.ascontiguousarray(np.where(glass_like(scene), ROUGHNESS, 0.))
        v = displacement(scene, LENGTH)
        say()
        say("%s (%dx%d, accel %d, %d primitives, %d glass-like, %d lights, view: yaw 10 degrees, no lens)"
            % (label, w, h, accel, scene.num_prims, int(glass_like(scene).sum()), len(scene.lights)))
        say("  %2s %-24s %9s %10s %10s %10s %8s" % ("s", "call", "wall ms", "ms_render", "ms_total", "kernel ms", "x lens"))
        try:
            for s in SAMPLES:
                ln = _abi.RmLens()
                ln.aperture, ln.focus, ln.samples = 0., 1., s

                def lens_call(st):
                    return L.rm_render_lens(hd, C.byref(p), C.byref(view), C.byref(ln), out, out8, C.byref(st) if st is not None else None)
                wall, ren0, tot = timed(lens_call)
                km = kernel_ms(lens_call, "lens_kernel")
                say("  %2d %-24s %9.3f %10.3f %10.3f %10.3f %8s" % (s, "rm_render_lens", wall, ren0, tot, km, "1.00"))
                al = _abi.RmAreaLights()
                al.n_lights, al.radius, al.samples = radii.shape[0], radii.ctypes.data_as(C.POINTER(C.c_double)), s
                rg = _abi.RmRoughGlass()
                rg.n_prims, rg.roughness, rg.samples = g.shape[0], g.ctypes.data_as(C.POINTER(C.c_double)), s
                mo = _abi.RmMotion()
                mo.n_prims, mo.displacement, mo.samples = v.shape[0], v.ctypes.data_as(C.POINTER(C.c_double)), s
                for which in SETS:
                    a = C.byref(al) if "area" in which else None
                    b = C.byref(rg) if "rough" in which else None
                    m = C.byref(mo) if "motion" in which else None

                    def dist_call(st, a=a, b=b, m=m):
                        return L.rm_render_distributed(hd, C.byref(p), s, C.byref(view), None, a, b, m, out, out8,
                                                       C.byref(st) if st is not None else None)
                    wall, ren, tot = timed(dist_call)
                    km = kernel_ms(dist_call, "distributed_kernel")
                    say("  %2d %-24s %9.3f %10.3f %10.3f %10.3f %8.2f" % (s, which, wall, ren, tot, km, ren / ren0))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("ms_render: device time of the traced and resolved rows (lens_kernel / distributed_kernel); ms_total: the whole call,")
    say("copies included; kernel ms: the kernel's mean time under torch.profiler; x lens: ms_render over rm_render_lens's at the")
    say("same s.  area: every light radius %g; rough: roughness %g on the glass-like primitives; motion: every shape moves by %g," % (RADIUS, ROUGHNESS, LENGTH))
    say("each in its own seeded direction (the hierarchy frames with motion walk the swept hierarchy).")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
