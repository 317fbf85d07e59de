"""Cost of diffuse interreflection (rm_render_indirect) on one GPU, next to rm_render_lens at the same s and view.

    python tools/indirect_bench.py [--out FILE] [--calls N]

For cornell_box at 3840x2160 (brute force), demo at 1600x1280 and stress_4k through the hierarchy (1024 spheres + 8192
triangles, 3840x2160, accel = 1), at s = 2 and 4 and max_depth 3 and 5, under a camera turned 10 degrees to the left (so that
rm_render_lens runs lens_kernel rather than routing to rm_render_supersampled) and without a lens: rm_render_lens and
rm_render_indirect, each the call's ms_render (device time of the traced and resolved rows, CUDA events), its ms_total
(device time of the whole call, copies included) and the host wall time around the synchronous call, medians of N calls after
two warm-up calls.  Outputs: float + 8-bit frame into pinned host memory (rm_host_alloc).  The card's name and power limit are
read in the same run (nvidia-smi --query-gpu, read-only)."""
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
from supersample_bench import card  # noqa: E402

# (label, description, width, height, accel)
CASES = [("cornell_4k", workloads.describe("cornell_box"), 3840, 2160, 0),
         ("demo", workloads.describe("demo"), 1600, 1280, 0),
         ("stress_4k_bvh", workloads.describe("stress", n_spheres=1024, grid=64), 3840, 2160, 1)]
SAMPLES = (2, 4)
DEPTHS = (3, 5)
YAW = math.radians(10.)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=5)
    args = ap.parse_args()
    import torch

    rm.init(0)
    L = _abi.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say("diffuse interreflection (rm_render_indirect), one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 2 warm-up calls; outputs: float + 8-bit frame into pinned host memory" % args.calls)
    view = _abi.RmView()
    view.forward[:] = [-math.sin(YAW), 0., -math.cos(YAW)]
    view.up[:] = [0., 1., 0.]
    for label, desc, w, h, accel in CASES:
        scene = workloads.build_scene(desc)
        hd = scene.device_handle()
        out = L.rm_host_alloc(h * w * 12)
        out8 = L.rm_host_alloc(h * w * 3)
        say()
        say("%s (%dx%d, accel %d, %d primitives, view: yaw 10 degrees, no lens)" % (label, w, h, accel, scene.num_prims))
        say("  %5s %2s %-20s %9s %10s %10s %8s" % ("depth", "s", "call", "wall ms", "ms_render", "ms_total", "x lens"))
        try:
            for depth in DEPTHS:
                r = rm.create_renderer(1.5, h, w)
                r.accel, r.max_depth = bool(accel), depth
                fb = rm.create_frame_buffer(32, 32)
                fb.width, fb.height = w, h
                p = r.params(fb, scene)
                for s in SAMPLES:
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

                    ln = _abi.RmLens()
                    ln.aperture, ln.focus, ln.samples = 0., 1., s

                    def lens_call(st):
                        return L.rm_render_lens(hd, C.byref(p), C.byref(view), C.byref(ln), out, out8, C.byref(st))

                    def indirect_call(st):
                        return L.rm_render_indirect(hd, C.byref(p), C.byref(view), None, s, out, out8, C.byref(st))
                    wall, ren0, tot = timed(lens_call)
                    say("  %5d %2d %-20s %9.3f %10.3f %10.3f %8s" % (depth, s, "rm_render_lens", wall, ren0, tot, "1.00"))
                    wall, ren, tot = timed(indirect_call)
                    say("  %5d %2d %-20s %9.3f %10.3f %10.3f %8.2f" % (depth, s, "rm_render_indirect", wall, ren, tot, ren / ren0))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("ms_render: device time of the traced and resolved rows (lens_kernel / indirect_kernel, CUDA events); ms_total: the")
    say("whole call, copies included; x lens: ms_render over rm_render_lens's at the same s and max_depth.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
