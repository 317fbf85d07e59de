"""Cost of camera orientation (rm_render_view) on one GPU.

    python tools/view_bench.py [--out FILE] [--calls N]

For cornell_4k (cornell_box 3840x2160), demo (1600x1280) and stress_4k through the hierarchy (1024 spheres + 8192 triangles,
3840x2160, accel = 1):
  * rm_render against rm_render_view with the identity view -- the same kernels: device time (K0 + K1, rm_set_profiling
    events) and call time (host wall time around the synchronous call), medians of N calls, the two alternated call by call;
  * the five views of the tests (yaw 30, pitch -20, roll 90, forward +x, straight down): device time, ray segments and device
    time per segment against the default view.  Segments: the instrumented kernel's closest + any-hit segments (one extra
    call with stats->pixels = 1) without the hierarchy, rendered pixels + rm_scene_query_count with it.
Outputs: float frame + primary ids into pinned host memory (rm_host_alloc), so that both calls take the same host path.
The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
import argparse
import ctypes as C
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import rusty_marcher_b200 as rm  # noqa: E402
from rusty_marcher_b200 import _abi, workloads  # noqa: E402
from rusty_marcher_b200.renderer import _view  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from supersample_bench import card  # noqa: E402

CASES = [("cornell_4k", workloads.describe("cornell_box"), 3840, 2160, 0),
         ("demo", workloads.describe("demo"), 1600, 1280, 0),
         ("stress_4k_bvh", workloads.describe("stress", n_spheres=1024, grid=64), 3840, 2160, 1)]
VIEWS = [("default", ((0., 0., -1.), (0., 1., 0.))),
         ("yaw30", ((-np.sin(np.radians(30.)), 0., -np.cos(np.radians(30.))), (0., 1., 0.))),
         ("pitch-20", ((0., -np.sin(np.radians(20.)), -np.cos(np.radians(20.))), (0., 1., 0.))),
         ("roll90", ((0., 0., -1.), (1., 0., 0.))),
         ("forward+x", ((1., 0., 0.), (0., 1., 0.))),
         ("down", ((0., -1., 0.), (0., 0., -1.)))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=30)
    args = ap.parse_args()
    import torch

    rm.init(0)
    L = _abi.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say("camera orientation (rm_render_view), one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 3 warm-up calls; outputs: float frame + primary ids into pinned host memory" % args.calls)
    _abi.check(L.rm_set_profiling(1))
    for label, desc, w, h, accel in CASES:
        scene = workloads.build_scene(desc)
        r = rm.create_renderer(1.5, h, w)
        r.accel = bool(accel)
        fb = rm.create_frame_buffer(32, 32)
        fb.width, fb.height = w, h
        p = r.params(fb, scene)
        hd = scene.device_handle()
        out = L.rm_host_alloc(h * w * 12)
        ids = L.rm_host_alloc(h * w * 4)
        pixels = (h // 32) * 32 * w
        try:
            def one(view):
                t0 = time.perf_counter()
                if view is None:
                    _abi.check(L.rm_render(hd, C.byref(p), out, ids, None, None))
                else:
                    _abi.check(L.rm_render_view(hd, C.byref(p), C.byref(view), out, ids, None, None))
                wall = 1e3 * (time.perf_counter() - t0)
                kp, kr = C.c_double(), C.c_double()
                _abi.check(L.rm_last_kernel_times(C.byref(kp), C.byref(kr)))
                return wall, kp.value + kr.value

            def timed(views):
                """medians of (call ms, device ms) per entry of `views`, the entries alternated call by call"""
                res = [[] for _ in views]
                for i in range(3 + args.calls):
                    for k, v in enumerate(views):
                        t = one(v)
                        if i >= 3:
                            res[k].append(t)
                return [(float(np.median([a for a, _ in x])), float(np.median([b for _, b in x]))) for x in res]

            def segments(view):
                if accel:
                    q = C.c_uint64()
                    _abi.check(L.rm_scene_query_count(hd, C.byref(q), 1))
                    _abi.check(L.rm_render_view(hd, C.byref(p), C.byref(view), out, ids, None, None))
                    _abi.check(L.rm_scene_query_count(hd, C.byref(q), 1))
                    return pixels + q.value
                st = _abi.RmStats()
                st.pixels = 1
                _abi.check(L.rm_render_view(hd, C.byref(p), C.byref(view), out, ids, None, C.byref(st)))
                return st.closest_segments + st.anyhit_segments

            say()
            say("%s (%dx%d, accel %d)" % (label, w, h, accel))
            (wa, da), (wb, db) = timed([None, _view(*VIEWS[0][1])])
            say("  rm_render                      call %8.3f ms   device %8.3f ms" % (wa, da))
            say("  rm_render_view, identity view  call %8.3f ms   device %8.3f ms   (%+.2f %% device)" % (wb, db, 100. * (db / da - 1.)))
            say("  %-10s %10s %12s %10s %12s" % ("view", "device ms", "segments", "ns/seg", "vs default"))
            base = None
            res = timed([_view(*v) for _, v in VIEWS])
            for (name, v), (_, dev) in zip(VIEWS, res):
                seg = segments(_view(*v))
                ns = 1e6 * dev / seg if seg else float("nan")
                if base is None:
                    base = ns
                say("  %-10s %10.3f %12d %10.4f %+11.1f%%" % (name, dev, seg, ns, 100. * (ns / base - 1.)))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(ids)
            scene.release()
    _abi.check(L.rm_set_profiling(0))
    say()
    say("device ms: K0 + K1 (rm_last_kernel_times); call ms: wall time of the synchronous call.  The default view is")
    say("rm_render_view's identity call, i.e. rm_render's own path.  segments: closest + any-hit ray segments of the frame")
    say("(instrumented kernel) without the hierarchy, rendered pixels + rm_scene_query_count with it.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
