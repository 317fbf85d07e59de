"""Cost of path-traced frames (rm_render_path) on one GPU, next to rm_render_distributed and rm_render_indirect at the same
settings.

    python tools/path_bench.py [--out FILE] [--calls N]

For cornell_box at 3840x2160 (brute force), demo at 1600x1280 and stress_4k through the hierarchy (1024 spheres + 8192
triangles, 3840x2160, accel = 1), at s = 2 and 4 and max_depth 3 and 5, under a camera turned 10 degrees to the left and
without a lens, for two combinations of effects: area lights alone (every light of radius 2), and area lights + rough glass
(roughness 0.1 on every glass-like primitive) + motion (every primitive moving by (0.5, 0.25, 0)).  rm_render_distributed and
rm_render_path take the effects; rm_render_indirect has none (its frame is the bounce alone).  Each call's ms_render (device
time of the traced and resolved rows, CUDA events), its ms_total (device time of the whole call, copies included) and the
host wall time around the synchronous call, medians of N calls after two warm-up calls.  Outputs: float + 8-bit frame into
pinned host memory (rm_host_alloc).  The card's name and power limit are read in the same run (nvidia-smi --query-gpu,
read-only)."""
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
COMBOS = ("area", "area+rough+motion")
YAW = math.radians(10.)


def glass_like_by_prim(scene):
    """is_glass_like by primitive id (shapes in scene order, an Obj once per triangle)."""
    from rusty_marcher_b200.obj import Obj
    out = []
    for s in scene.shapes:
        if isinstance(s, Obj):
            out.extend(float(f) for f in s.reflectances["is_glass_like"])
        else:
            out.append(float(s.reflectance.is_glass_like))
    return np.array(out)


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

    say("path-traced frames (rm_render_path), one GPU: %s" % torch.cuda.get_device_name(0))
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
        radii = np.full(len(scene.lights), 2.)
        rough = np.ascontiguousarray(0.1 * glass_like_by_prim(scene))
        disp = np.ascontiguousarray(np.tile([0.5, 0.25, 0.], (scene.num_prims, 1)))
        say()
        say("%s (%dx%d, accel %d, %d primitives, %d glass-like, view: yaw 10 degrees, no lens)"
            % (label, w, h, accel, scene.num_prims, int((rough > 0).sum())))
        say("  %-17s %5s %2s %-22s %9s %10s %10s %7s %7s" % ("effects", "depth", "s", "call", "wall ms", "ms_render", "ms_total",
                                                            "x dist", "x ind"))
        try:
            for combo in COMBOS:
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

                        lights = _abi.RmAreaLights()
                        lights.n_lights, lights.radius, lights.samples = radii.shape[0], radii.ctypes.data_as(C.POINTER(C.c_double)), s
                        rg = mo = None
                        if "rough" in combo:
                            rg = _abi.RmRoughGlass()
                            rg.n_prims, rg.roughness, rg.samples = rough.shape[0], rough.ctypes.data_as(C.POINTER(C.c_double)), s
                        if "motion" in combo:
                            mo = _abi.RmMotion()
                            mo.n_prims, mo.displacement, mo.samples = disp.shape[0], disp.ctypes.data_as(C.POINTER(C.c_double)), s
                        ref = lambda x: C.byref(x) if x is not None else None     # noqa: E731

                        def dist_call(st):
                            return L.rm_render_distributed(hd, C.byref(p), s, C.byref(view), None, C.byref(lights), ref(rg), ref(mo),
                                                           out, out8, C.byref(st))

                        def indirect_call(st):
                            return L.rm_render_indirect(hd, C.byref(p), C.byref(view), None, s, out, out8, C.byref(st))

                        def path_call(st):
                            return L.rm_render_path(hd, C.byref(p), s, C.byref(view), None, C.byref(lights), ref(rg), ref(mo), out, out8,
                                                    C.byref(st))
                        row = "  %-17s %5d %2d %-22s %9.3f %10.3f %10.3f %7s %7s"
                        wall, ren_d, tot = timed(dist_call)
                        say(row % (combo, depth, s, "rm_render_distributed", wall, ren_d, tot, "", ""))
                        wall, ren_i, tot = timed(indirect_call)
                        say(row % (combo, depth, s, "rm_render_indirect", wall, ren_i, tot, "", ""))
                        wall, ren, tot = timed(path_call)
                        say(row % (combo, depth, s, "rm_render_path", wall, ren, tot, "%.2f" % (ren / ren_d), "%.2f" % (ren / ren_i)))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("ms_render: device time of the traced and resolved rows (distributed_kernel / indirect_kernel / path_kernel, CUDA")
    say("events); ms_total: the whole call, copies included; x dist, x ind: rm_render_path's ms_render over")
    say("rm_render_distributed's and rm_render_indirect's at the same s, max_depth and effects.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
