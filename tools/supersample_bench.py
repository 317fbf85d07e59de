"""Cost of supersampled anti-aliasing (rm_render_supersampled) on one GPU.

    python tools/supersample_bench.py [--out FILE] [--calls N]

For cornell_4k (cornell_box 3840x2160), cornell_1080p (1920x1080) and demo (1600x1280), at s = 1, 2 and 4:
  * ms per call: host wall time around the synchronous call (median of N), and the call's own ms_render (render kernels of
    the s x frame) and ms_total (device time of the whole call, copies included);
  * rm_render on the same frame with the same two outputs (float and 8-bit frame), for the s = 1 comparison;
  * in a separate pass under torch.profiler (CUDA activities): the mean time of resolve_box_kernel, its achieved bytes/s --
    12 s^2 bytes read and 12 written per output pixel -- and its share of the 7.7 TB/s data-sheet HBM bandwidth of a B200,
    and its share of ms_total.
The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).  Output buffers are pinned host
memory (rm_host_alloc).  The s x frame is 12 s^2 W rows bytes (1.6 GB at 4K, s = 4): from s = 2 at 4K it exceeds the 126 MB L2,
so the resolve reads HBM; at 1080p s = 2 (97 MB) part of it may still sit in L2 from the render kernel."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import rusty_marcher_b200 as rm  # noqa: E402
from rusty_marcher_b200 import _abi, workloads  # noqa: E402

HBM_BYTES_PER_S = 7.7e12                                       # B200 data sheet (one GPU of an HGX B200)
CASES = [("cornell_4k", "cornell_box", 3840, 2160), ("cornell_1080p", "cornell_box", 1920, 1080), ("demo", "demo", 1600, 1280)]
SAMPLES = (1, 2, 4)


def card():
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q + ": " + r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "nvidia-smi unavailable: %s" % e


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

    say("supersampled anti-aliasing, one GPU: %s" % torch.cuda.get_device_name(0))
    say("card: %s" % card())
    say("calls per point: %d (median), after 3 warm-up calls; outputs: float + 8-bit frame into pinned host memory" % args.calls)
    say()
    say("%-14s %2s %9s %10s %10s %10s %11s %9s %9s %8s" % ("workload", "s", "wall ms", "ms_render", "ms_total", "resolve us",
                                                          "resolve GB", "TB/s", "of HBM", "of total"))
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

            wall, ren, tot = timed(lambda st: L.rm_render(hd, C.byref(p), out, None, out8, C.byref(st)))
            say("%-14s %2s %9.3f %10.3f %10.3f   (rm_render, same outputs)" % (label, "-", wall, ren, tot))
            for s in SAMPLES:
                wall, ren, tot = timed(lambda st: L.rm_render_supersampled(hd, C.byref(p), s, out, out8, C.byref(st)))
                # the resolve kernel alone, in a pass of its own under the profiler
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        _abi.check(L.rm_render_supersampled(hd, C.byref(p), s, out, out8, None))
                    torch.cuda.synchronize()
                ks = [e.time_range.elapsed_us() for e in prof.events() if "resolve_box_kernel" in e.name and e.device_type.name == "CUDA"]
                if not ks:                                      # (kernels attached to a host-side event instead)
                    ks = [k.duration for e in prof.events() for k in getattr(e, "kernels", []) if "resolve_box_kernel" in k.name]
                if len(ks) != 5:
                    raise RuntimeError("torch.profiler recorded %d resolve_box_kernel launches, expected 5" % len(ks))
                us = float(np.mean(ks))
                nbytes = (12 * s * s + 12) * w * rows
                rate = nbytes / (us * 1e-6)
                say("%-14s %2d %9.3f %10.3f %10.3f %10.1f %11.3f %9.2f %8.1f%% %7.1f%%" % (
                    label, s, wall, ren, tot, us, nbytes / 1e9, rate / 1e12, 100 * rate / HBM_BYTES_PER_S, 100 * us * 1e-3 / tot))
        finally:
            L.rm_host_free(out)
            L.rm_host_free(out8)
            scene.release()
    say()
    say("resolve GB: bytes the resolve must move (12 s^2 read + 12 written per output pixel); TB/s: those over its mean kernel time;")
    say("of HBM: that over 7.7 TB/s (data sheet, not a measured peak); of total: resolve time over the call's median ms_total.")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
