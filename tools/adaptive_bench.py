"""Cost and quality of adaptive anti-aliasing (rm_render_adaptive) against full supersampling on one GPU.

    python tools/adaptive_bench.py [--out FILE] [--calls N]

For cornell_4k (cornell_box 3840x2160), cornell_1080p (1920x1080) and demo (1600x1280), at s = 2 and 4, for the default
contrast of Renderer.render_adaptive, +inf (geometric edges only) and -1 (every pixel):
  * the refined fraction of the output rows;
  * ms per call: host wall time around the synchronous call (median of N), ms_render (device time from the 1x render to the
    resolved float rows) and ms_total (the whole call, copies included);
  * rm_render_supersampled at the same point: its ms_render plus its resolve kernel (its ms_render covers the s x render
    only), and its ms_total, medians the same way;
  * in a separate pass under torch.profiler (CUDA activities): the mean times of adaptive_mark_kernel,
    adaptive_subpixel_kernel and adaptive_resolve_kernel, and of resolve_box_kernel for the supersampled call;
  * quality against rm_render_supersampled: the share of pixels whose 8-bit value differs from it by more than 1 LSB in some
    channel, and the largest difference.
Outputs as tools/supersample_bench.py: float + 8-bit frame into pinned host memory (rm_host_alloc), plus the mask for the
adaptive call.  The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
import argparse
import ctypes as C
import inspect
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import rusty_marcher_b200 as rm  # noqa: E402
from rusty_marcher_b200 import _abi, workloads  # noqa: E402
from rusty_marcher_b200.renderer import Renderer  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from supersample_bench import card  # noqa: E402

CASES = [("cornell_4k", "cornell_box", 3840, 2160), ("cornell_1080p", "cornell_box", 1920, 1080), ("demo", "demo", 1600, 1280)]
SAMPLES = (2, 4)
DEFAULT_CONTRAST = inspect.signature(Renderer.render_adaptive).parameters["contrast"].default
CONTRASTS = (DEFAULT_CONTRAST, float("inf"), -1.)
KERNELS = ("adaptive_mark_kernel", "adaptive_subpixel_kernel", "adaptive_resolve_kernel", "resolve_box_kernel")


def kernel_means(prof, n):
    """Mean device time (us) per kernel name of KERNELS over the n calls of a profiled pass (0 when a kernel did not run)."""
    out = {}
    for name in KERNELS:
        ks = [e.time_range.elapsed_us() for e in prof.events() if name in e.name and e.device_type.name == "CUDA"]
        if not ks:                                              # (kernels attached to a host-side event instead)
            ks = [k.duration for e in prof.events() for k in getattr(e, "kernels", []) if name in k.name]
        if ks and len(ks) != n:
            raise RuntimeError("torch.profiler recorded %d %s launches, expected %d" % (len(ks), name, n))
        out[name] = float(np.mean(ks)) if ks else 0.
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    rm.init(0)
    L = _abi.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say("adaptive anti-aliasing against full supersampling, one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 3 warm-up calls; outputs: float + 8-bit frame (+ mask) into pinned host memory" % args.calls)
    say("default contrast (Renderer.render_adaptive): %g" % DEFAULT_CONTRAST)
    say()
    say("%-14s %2s %8s %8s | %8s %9s %9s | %9s %9s | %8s %8s %8s | %7s %4s" % (
        "workload", "s", "contrast", "refined", "wall ms", "ms_render", "ms_total", "SS ren+rs", "SS total",
        "mark us", "sub us", "res us", ">1 LSB", "max"))
    for label, name, w, h in CASES:
        scene = workloads.scene(name)
        r = rm.create_renderer(1.5, h, w)
        fb = rm.create_frame_buffer(32, 32)
        fb.width, fb.height = w, h
        p = r.params(fb, scene)
        hd = scene.device_handle()
        rows = (h // 32) * 32
        out = L.rm_host_alloc(h * w * 12)
        out8 = L.rm_host_alloc(h * w * 3)
        outm = L.rm_host_alloc(h * w)
        ss8 = np.zeros((h, w, 3), dtype=np.uint8)
        try:
            def timed(fn):
                st = _abi.RmStats()
                walls, ren, tot = [], [], []
                for i in range(3 + args.calls):
                    t0 = time.perf_counter()
                    _abi.check(fn(st))
                    t1 = time.perf_counter()
                    if i >= 3:
                        walls.append(1e3 * (t1 - t0))
                        ren.append(st.ms_render)
                        tot.append(st.ms_total)
                return float(np.median(walls)), float(np.median(ren)), float(np.median(tot))

            def profiled(fn, n=5):
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(n):
                        _abi.check(fn())
                    torch.cuda.synchronize()
                return kernel_means(prof, n)

            for s in SAMPLES:
                _, ss_ren, ss_tot = timed(lambda st: L.rm_render_supersampled(hd, C.byref(p), s, out, out8, C.byref(st)))
                ss_res = profiled(lambda: L.rm_render_supersampled(hd, C.byref(p), s, out, out8, None))["resolve_box_kernel"]
                C.memmove(ss8.ctypes.data, out8, h * w * 3)
                for contrast in CONTRASTS:
                    fn = lambda st: L.rm_render_adaptive(hd, C.byref(p), s, contrast, out, out8, outm, C.byref(st))  # noqa: E731
                    wall, ren, tot = timed(fn)
                    km = profiled(lambda: L.rm_render_adaptive(hd, C.byref(p), s, contrast, out, out8, outm, None))
                    got8 = np.ctypeslib.as_array(C.cast(out8, C.POINTER(C.c_uint8)), shape=(h, w, 3))[:rows]
                    mask = np.ctypeslib.as_array(C.cast(outm, C.POINTER(C.c_uint8)), shape=(h, w))[:rows]
                    d = np.abs(got8.astype(np.int16) - ss8[:rows].astype(np.int16)).max(axis=2)
                    say("%-14s %2d %8g %7.2f%% | %8.3f %9.3f %9.3f | %9.3f %9.3f | %8.1f %8.1f %8.1f | %6.3f%% %4d" % (
                        label, s, contrast, 100. * mask.mean(), wall, ren, tot, ss_ren + 1e-3 * ss_res, ss_tot,
                        km["adaptive_mark_kernel"], km["adaptive_subpixel_kernel"], km["adaptive_resolve_kernel"],
                        100. * (d > 1).mean(), int(d.max())))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            L.rm_host_free(outm)
            scene.release()
    say()
    say("refined: share of the output rows' pixels supersampled; wall ms / ms_render / ms_total: rm_render_adaptive (ms_render:")
    say("1x render + mark + sub-pixel rays + resolve); SS ren+rs: rm_render_supersampled's ms_render (its s x render) plus its")
    say("resolve_box_kernel, SS total: its ms_total; mark / sub / res us: mean kernel times under torch.profiler;")
    say(">1 LSB / max: pixels whose 8-bit value differs from rm_render_supersampled's by more than 1 in some channel, and the")
    say("largest difference (each frame tone-mapped by its own maximum).")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
