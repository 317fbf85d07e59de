"""Cost of depth of field (rm_render_lens) on one GPU, next to rm_render_supersampled at the same s.

    python tools/lens_bench.py [--out FILE] [--calls N]

For cornell_4k (cornell_box 3840x2160), demo (1600x1280) and stress_4k through the hierarchy (1024 spheres + 8192 triangles,
3840x2160, accel = 1), at s = 2 and 4:
  * rm_render_supersampled, and rm_render_lens with the aperture at 0 (routed to rm_render_supersampled), small and large:
    call time (host wall time around the synchronous call), the call's ms_render (device time from the start of the render
    to the resolved rows) and ms_total (device time of the whole call, copies included), medians of N calls;
  * in a separate pass under torch.profiler (CUDA activities): the mean time of lens_kernel;
  * device time per ray segment: ms_render over the closest-hit + any-hit segments of the supersampled frame at the same s
    -- the instrumented kernel's counts on the s x frame without the hierarchy, its sample rays + rm_scene_query_count with
    it.  The lens frame traces as many sample rays; its secondary and shadow segments differ from those only where the blur
    moves a sample onto another surface, so the same count is used as the denominator of both.
Outputs: float + 8-bit frame into pinned host memory (rm_host_alloc).  The card's name and power limit are read in the same
run (nvidia-smi --query-gpu, read-only)."""
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

# (label, description, width, height, accel, focus, small aperture, large aperture)
CASES = [("cornell_4k", workloads.describe("cornell_box"), 3840, 2160, 0, 300., 2., 10.),
         ("demo", workloads.describe("demo"), 1600, 1280, 0, 12., 0.1, 0.5),
         ("stress_4k_bvh", workloads.describe("stress", n_spheres=1024, grid=64), 3840, 2160, 1, 100., 0.5, 2.)]
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

    say("depth of field (rm_render_lens), one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 2 warm-up calls; outputs: float + 8-bit frame into pinned host memory" % args.calls)
    for label, desc, w, h, accel, focus, small, large in CASES:
        scene = workloads.build_scene(desc)
        r = rm.create_renderer(1.5, h, w)
        r.accel = bool(accel)
        fb = rm.create_frame_buffer(32, 32)
        fb.width, fb.height = w, h
        p = r.params(fb, scene)
        hd = scene.device_handle()
        rows = (h // 32) * 32
        out = L.rm_host_alloc(h * w * 12)
        out8 = L.rm_host_alloc(h * w * 3)
        say()
        say("%s (%dx%d, accel %d, focus %g)" % (label, w, h, accel, focus))
        say("  %2s %-22s %9s %10s %10s %10s %14s %9s" % ("s", "call", "wall ms", "ms_render", "ms_total", "kernel ms", "segments", "ns/seg"))
        try:
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

                def kernel_ms(fn, name):
                    torch.cuda.synchronize()
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        for _ in range(3):
                            _abi.check(fn(None))
                        torch.cuda.synchronize()
                    ks = [e.time_range.elapsed_us() for e in prof.events() if name in e.name and e.device_type.name == "CUDA"]
                    if not ks:                                  # (kernels attached to a host-side event instead)
                        ks = [k.duration for e in prof.events() for k in getattr(e, "kernels", []) if name in k.name]
                    if len(ks) != 3:
                        raise RuntimeError("torch.profiler recorded %d %s launches, expected 3" % (len(ks), name))
                    return 1e-3 * float(np.mean(ks))

                # ray segments of the supersampled frame
                sp = _abi.RmParams.from_buffer_copy(p)
                sp.width, sp.height = s * w, s * h
                sp.patch_row_begin, sp.patch_row_end = 0, s * (h // 32)
                if accel:
                    q = C.c_uint64()
                    _abi.check(L.rm_scene_query_count(hd, C.byref(q), 1))
                    _abi.check(L.rm_render_supersampled(hd, C.byref(p), s, out, out8, None))
                    _abi.check(L.rm_scene_query_count(hd, C.byref(q), 1))
                    seg = s * s * rows * w + q.value
                else:
                    sub = L.rm_host_alloc(s * s * h * w * 12)
                    try:
                        st = _abi.RmStats()
                        st.pixels = 1
                        _abi.check(L.rm_render(hd, C.byref(sp), sub, None, None, C.byref(st)))
                        seg = st.closest_segments + st.anyhit_segments
                    finally:
                        L.rm_host_free(sub)

                def ss_call(st):
                    return L.rm_render_supersampled(hd, C.byref(p), s, out, out8, C.byref(st) if st is not None else None)
                wall, ren, tot = timed(ss_call)
                say("  %2d %-22s %9.3f %10.3f %10.3f %10s %14d %9.4f" % (s, "rm_render_supersampled", wall, ren, tot, "-", seg, 1e6 * ren / seg))
                for tag, a in (("lens, aperture 0", 0.), ("lens, aperture %g" % small, small), ("lens, aperture %g" % large, large)):
                    ln = _abi.RmLens()
                    ln.aperture, ln.focus, ln.samples = a, focus, s

                    def lens_call(st, ln=ln):
                        return L.rm_render_lens(hd, C.byref(p), None, C.byref(ln), out, out8, C.byref(st) if st is not None else None)
                    wall, ren, tot = timed(lens_call)
                    km = kernel_ms(lens_call, "lens_kernel") if a > 0 else float("nan")
                    say("  %2d %-22s %9.3f %10.3f %10.3f %10s %14d %9.4f" % (s, tag, wall, ren, tot, "-" if a == 0 else "%.3f" % km, seg,
                                                                            1e6 * ren / seg))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("ms_render: device time of the traced and resolved rows (rm_render_supersampled: the s x frame's K0 + K1 and the resolve;")
    say("rm_render_lens: lens_kernel); ms_total: the whole call, copies included; kernel ms: lens_kernel's mean time under")
    say("torch.profiler.  Aperture 0 without a view is rm_render_supersampled's frame: the call is routed there.  segments: closest")
    say("+ any-hit ray segments of the supersampled frame at the same s (see the module docstring); ns/seg: ms_render over them.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
