"""Cost of soft shadows (rm_render_area_lights) on one GPU, next to rm_render on the same scene.

    python tools/area_bench.py [--out FILE] [--calls N]

For cornell_4k (cornell_box 3840x2160), demo (1600x1280) and stress_4k through the hierarchy (1024 spheres + 8192 triangles,
3840x2160, accel = 1), rm_render and rm_render_area_lights at s = 2 and 4, every light given the same radius, small and
large:
  * call time (host wall time around the synchronous call), the call's ms_render (device time of the rendered rows: K0 + K1
    for rm_render, K0 + area_light_kernel for the area lights) and ms_total (device time of the whole call, copies
    included), medians of N calls, and ms_render against rm_render's;
  * in a separate pass under torch.profiler (CUDA activities): the mean time of area_light_kernel.
Outputs: float + primary ids + 8-bit frame into pinned host memory (rm_host_alloc), for both calls.  The card's name and power
limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
import argparse
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import rusty_marcher_b200 as rm  # noqa: E402
from rusty_marcher_b200 import _abi, workloads  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from supersample_bench import card  # noqa: E402

# (label, description, width, height, accel, small radius, large radius)
CASES = [("cornell_4k", workloads.describe("cornell_box"), 3840, 2160, 0, 2., 10.),
         ("demo", workloads.describe("demo"), 1600, 1280, 0, 0.5, 3.),
         ("stress_4k_bvh", workloads.describe("stress", n_spheres=1024, grid=64), 3840, 2160, 1, 0.5, 3.)]
SAMPLES = (2, 4)


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

    say("soft shadows (rm_render_area_lights), one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 2 warm-up calls; outputs: float + ids + 8-bit frame into pinned host memory" % args.calls)
    for label, desc, w, h, accel, small, large in CASES:
        scene = workloads.build_scene(desc)
        r = rm.create_renderer(1.5, h, w)
        r.accel = bool(accel)
        fb = rm.create_frame_buffer(32, 32)
        fb.width, fb.height = w, h
        p = r.params(fb, scene)
        hd = scene.device_handle()
        n_lights = len(scene.lights)
        out = L.rm_host_alloc(h * w * 12)
        ids = L.rm_host_alloc(h * w * 4)
        out8 = L.rm_host_alloc(h * w * 3)
        say()
        say("%s (%dx%d, accel %d, %d lights)" % (label, w, h, accel, n_lights))
        say("  %2s %-24s %9s %10s %10s %10s %8s" % ("s", "call", "wall ms", "ms_render", "ms_total", "kernel ms", "x render"))
        try:
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
                if not ks:                                      # (kernels attached to a host-side event instead)
                    ks = [k.duration for e in prof.events() for k in getattr(e, "kernels", []) if name in k.name]
                if len(ks) != 3:
                    raise RuntimeError("torch.profiler recorded %d %s launches, expected 3" % (len(ks), name))
                return 1e-3 * float(np.mean(ks))

            def render_call(st):
                return L.rm_render(hd, C.byref(p), out, ids, out8, C.byref(st) if st is not None else None)
            wall, base, tot = timed(render_call)
            say("  %2s %-24s %9.3f %10.3f %10.3f %10s %8s" % ("-", "rm_render", wall, base, tot, "-", "1.00"))
            for s in SAMPLES:
                for radius in (small, large):
                    radii = (C.c_double * n_lights)(*([radius] * n_lights))
                    al = _abi.RmAreaLights()
                    al.n_lights, al.radius, al.samples = n_lights, C.cast(radii, C.POINTER(C.c_double)), s

                    def area_call(st, al=al):
                        return L.rm_render_area_lights(hd, C.byref(p), C.byref(al), out, ids, out8, C.byref(st) if st is not None else None)
                    wall, ren, tot = timed(area_call)
                    km = kernel_ms(area_call, "area_light_kernel")
                    say("  %2d %-24s %9.3f %10.3f %10.3f %10.3f %8.2f" % (s, "area lights, radius %g" % radius, wall, ren, tot, km, ren / base))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(ids)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("ms_render: device time of the rendered rows (rm_render: K0 + K1; rm_render_area_lights: K0 + area_light_kernel);")
    say("ms_total: the whole call, copies included; kernel ms: area_light_kernel's mean time under torch.profiler; x render:")
    say("ms_render over rm_render's on the same scene.  Every light of the scene has the radius given; s x s samples each.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
