#!/usr/bin/env python
"""bench.py -- ray segments/s and ms/frame of the render hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Workload (config.workload): the cornell_box mesh at 3840x2160, fov 1.5, camera origin, depth cap 3
-- the configuration BASELINE.json's metric and north_star target are quoted on (configs[2]; the
cornell_box2.obj it names does not exist in the reference, SURVEY.md fact 7).  A step is one frame
through rm_render_frame: K0 (per-frame records + tile schedule) and K1 (render, channel max, the
exchange over NVLink peer memory, fused normalise + quantise), one CUDA graph launch; with N > 1
GPUs the frame's 67 patch rows are dealt round-robin, one process per GPU (scaling "strong").
Every run also proves that the frame the ranks assemble IS the single-GPU frame (frame_matches_n1),
times the end-to-end call through host buffers (e2e: at N > 1 into ONE frame shared by the ranks)
and adds a short `heavy` leg on BASELINE.json's configs[4] at full size through the hierarchy.

`--impl reference` times the reference's own CPU algorithm (the f64 oracle restatement of the Rayon
patch loop -- the Rust original cannot be built here) on the host cores, same workload and metric.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ray_segments_per_s"
UNIT = "segments/s"
WORKLOADS = {
    # name: (scene, width, height, max_depth, scene kwargs)
    "cornell_4k": ("cornell_box", 3840, 2160, 3, {}),
    "cornell_1080p": ("cornell_box", 1920, 1080, 3, {}),
    "demo": ("demo", 1600, 1280, 3, {}),
    "dodecahedron_4k": ("dodecahedron", 3840, 2160, 3, {}),
    "stress_small": ("stress", 1920, 1080, 6, dict(n_spheres=512, grid=32)),
    # BASELINE.json configs[4] scaled to fit a bench run (1024 spheres + 8192 triangles instead of 4096 + 100,352, 4K instead
    # of 8K, same generator and depth cap 6): brute force over ~9k primitives per segment, ~0.1-0.2 s per frame on one GPU
    # -- the regime in which the row-band split can be expected to scale
    "stress_4k": ("stress", 3840, 2160, 6, dict(n_spheres=1024, grid=64)),
    # the same frame with RmParams.accel = 1: scene queries walk the bounding-volume hierarchy (SURVEY.md 8f row 4) instead
    # of every primitive -- bit-identical frame, O(log n) tests per segment.  Reported separately: the algorithmic work of
    # SURVEY.md 8d is defined by the reference's brute-force traversal, which this mode does not execute.
    "stress_4k_bvh": ("stress", 3840, 2160, 6, dict(n_spheres=1024, grid=64, accel=True)),
    # BASELINE.json configs[4] at full size: 4096 spheres + 100,352 triangles, 7680x4320, depth cap 6
    "stress_8k_bvh": ("stress", 7680, 4320, 6, dict(n_spheres=4096, grid=224, accel=True)),
}


def workload_of(name):
    """(scene, width, height, max_depth, scene kwargs, accel)"""
    scene, w, h, depth, kw = WORKLOADS[name]
    kw = dict(kw)
    accel = bool(kw.pop("accel", False))
    return scene, w, h, depth, kw, accel


def n_prims_of(desc):
    from rusty_marcher_b200 import workloads
    return workloads.n_prims(desc)


def config_of(args, extra=None):
    scene, w, h, depth, kw, accel = workload_of(args.workload)
    cfg = {"workload": "%s%s %dx%d fov 1.5 camera origin depth-cap %d (reference semantics: rows >= floor(H/32)*32 not rendered)"
                       % (scene, " " + json.dumps(kw, sort_keys=True) if kw else "", w, h, depth),
           "width": w, "height": h, "max_depth": depth, "scene": scene,
           "accel": "bvh (RmParams.accel = 1)" if accel else "none (the reference's brute-force traversal)"}
    if extra:
        cfg.update(extra)
    return cfg


class ClockSampler:
    """SM clock / clock-event (throttle) reasons during the timed region (B200_PROFILING.md's clocks line).

    Sampled in-process through NVML (nvidia_ml_py) from a thread every ~2 ms -- `nvidia-smi -lms` needs ~100 ms to come
    up and delivers one or two lines in a region this short; it is kept as the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.thread = index, None, None
        self.sm, self.mx, self.reasons, self.busy = [], [], set(), []
        self._stop = threading.Event()

    def _nvml_loop(self, nv, h):
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                 ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown))
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for name, bit in names:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:               # one failed query must not end the sampling
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: map the CUDA ordinal through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.index
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
            self.source = "nvml, 2 ms period"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.source = "nvidia-smi -lms 20"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=1.0)
        elif self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            for line in self.proc.communicate()[0].splitlines():
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    self.sm.append(float(f[1]))
                    self.mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower() == "active":
                        self.reasons.add(name)
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        sm, mx = self.sm, self.mx
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(self.reasons), "samples": len(sm),
                "source": self.source}


def cpu_reference_frame_time(desc, w, h, depth, budget_s, reps):
    """Times the oracle's Rayon-analogue patch loop (all host threads, uninstrumented).  Returns
    (seconds for a FULL frame, threads, sample description); strided patch sampling keeps it bounded."""
    from oracle import oracle as O
    from tests.oracle_scenes import build_oracle_scene
    import numpy as np
    osc = build_oracle_scene(desc)
    threads = O.hardware_threads()
    out = np.zeros((h, w, 3), dtype=np.float64)
    n_patches = (h // 32) * (w // 32)
    # calibrate on every 16th patch -- on fewer when pixels x primitives says the brute-force frame takes minutes (the
    # reference tests every primitive for every segment: configs[4] is ~3e12 primary tests alone)
    cal, max_stride = 16, 64
    while w * h * n_prims_of(desc) / cal > 4e9 and cal < 1024:
        cal *= 2
        max_stride = 1024
    t0 = time.perf_counter()
    O.render(osc, w, h, max_depth=depth, threads=threads, patch_stride=cal, want_ids=False, want_fragile=False, want_counters=False, out=out)
    full_est = (time.perf_counter() - t0) * cal
    stride = 1
    while full_est / stride * reps > budget_s and stride < max_stride:
        stride *= 2
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        O.render(osc, w, h, max_depth=depth, threads=threads, patch_stride=stride, want_ids=False, want_fragile=False, want_counters=False, out=out)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    n_sampled = len(range(0, n_patches, stride))
    full = best * n_patches / n_sampled
    sample = "best of %d passes over %d of %d 32x32 patches (every %d%s), %d threads, f64 restatement of the Rayon loop" % (
        reps, n_sampled, n_patches, stride, "th, extrapolated" if stride > 1 else "", threads)
    return full, threads, sample


def oracle_segments(desc, w, h, depth):
    """Segments of one frame from the oracle's counters (reference arm only)."""
    from oracle import oracle as O
    from tests.oracle_scenes import build_oracle_scene
    stride = 1
    while w * h * n_prims_of(desc) / stride > 1e10 and stride < 1024:
        stride *= 2                     # a frame the oracle cannot finish in minutes: count a patch sample and scale it
    r = O.render(build_oracle_scene(desc), w, h, max_depth=depth, patch_stride=stride, want_ids=False, want_fragile=False, want_counters=True)
    c = r["counters"]
    n_patches = (h // 32) * (w // 32)
    return int((c["closest_segments"] + c["anyhit_segments"]) * n_patches / len(range(0, n_patches, stride)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from rusty_marcher_b200 import workloads
    scene, w, h, depth, kw, _accel = workload_of(args.workload)
    desc = workloads.describe(scene, **kw)
    segs = oracle_segments(desc, w, h, depth)
    # one "step" = one (possibly patch-sampled) frame; keep the whole run within a few minutes
    total_steps = args.steps + args.warmup
    heavy = w * h * n_prims_of(desc) > 6.4e10       # minutes per brute-force frame: one bounded estimation pass only
    full, threads, sample = cpu_reference_frame_time(desc, w, h, depth, budget_s=min(150.0 / max(total_steps, 1) * 3, 60.0 if heavy else 1e9),
                                                     reps=1 if heavy else 3)
    from oracle import oracle as O
    from tests.oracle_scenes import build_oracle_scene
    import numpy as np
    osc = build_oracle_scene(desc)
    out = np.zeros((h, w, 3), dtype=np.float64)
    n_patches = (h // 32) * (w // 32)
    stride = 1
    while full / stride * total_steps > 150.0 and stride < (1024 if heavy else 64):
        stride *= 2
    n_sampled = len(range(0, n_patches, stride))
    times = []
    for i in range(total_steps):
        t0 = time.perf_counter()
        O.render(osc, w, h, max_depth=depth, threads=threads, patch_stride=stride, want_ids=False, want_fragile=False, want_counters=False, out=out)
        if i >= args.warmup:
            times.append((time.perf_counter() - t0) * n_patches / n_sampled)
    ms = 1e3 * sum(times) / len(times)
    value = segs / (ms * 1e-3)
    sample = "each step renders %d of %d 32x32 patches (every %d%s) with %d host threads; f64 C++ restatement of the reference's Rayon loop (Rust toolchain absent)" % (
        n_sampled, n_patches, stride, "th, time extrapolated to the frame" if stride > 1 else "", threads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": config_of(args, {"segments_per_frame": segs,
                                       "accel": "none: this arm is the reference's brute-force traversal (shapes.rs:92-143), whatever the workload's own arm uses"}),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


VERIFY_CAMERAS = {"default": [(0., 0., 0.), (30., -20., 10.), (-45., 15., 0.)],
                  "stress": [(0., 0., 0.), (7.5, -3.25, 20.), (-5., 2., -10.)]}


def verify_frames(tr, backend, cameras, world, rank, dev):
    """Driver-visible proof that the frame the ranks assemble is the single-GPU frame (SURVEY.md 8e; the reference's
    reassembly is engine/src/renderer.rs:92-108).  For each camera, back to back (consecutive frames alternate between
    rank 0's two 8-bit buffers, and rank 0 clears the other ranks' bands of the NEXT buffer inside the kernel): one frame
    through the product path at N ranks -- rm_render_frame, exchange inside the kernel -- then rank 0 renders the same
    frame alone (rm_render_device over every patch row + rm_tonemap_device, no exchange) and compares (1) the assembled
    RGB8 frame byte for byte and (2) the float rows of every rank, gathered once, bit for bit.  Outside every timed region.
    Returns (ok, sha256 of the first assembled 8-bit frame, detail) on rank 0, (True, None, None) elsewhere."""
    import ctypes as C
    import hashlib
    import torch
    import torch.distributed as dist
    from rusty_marcher_b200 import _abi, tiled
    L = backend.L
    h, w, n_patch = tr.height, tr.width, tr.n_patch_rows
    rows = n_patch * 32
    ok, sha, detail = True, None, []
    frames8, floats = [], []
    for cam in cameras:                                      # the product path, consecutive frames
        tr.set_camera(cam)
        f = tr.render()
        if rank == 0:
            frames8.append(f.clone())                        # stream-ordered: valid until the next frame is issued
        first = [tiled.bands_of(n_patch, r, world)[0] for r in range(world)]      # first band of every rank
        mine = tr.rgb[:rows].view(n_patch, 32, w, 3)[first[rank]::world].contiguous()
        if world == 1:
            floats.append(tr.rgb.clone())
        elif rank == 0:
            full = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
            fv = full[:rows].view(n_patch, 32, w, 3)
            fv[first[0]::world] = mine
            for r in range(1, world):
                n = len(range(first[r], n_patch, world))
                if n:
                    buf = torch.empty((n, 32, w, 3), dtype=torch.float32, device=dev)
                    dist.recv(buf, src=r)
                    fv[first[r]::world] = buf
            floats.append(full)
        elif mine.shape[0]:
            dist.send(mine, dst=0)
    torch.cuda.synchronize()
    if tr.peer is not None:
        tr.peer.status()
    if rank == 0:
        ref = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
        ref8 = torch.zeros((h, w, 3), dtype=torch.uint8, device=dev)
        smax = torch.zeros(1, dtype=torch.float32, device=dev)
        p = backend.frame_params((0, n_patch))
        stream = torch.cuda.current_stream().cuda_stream
        for i, cam in enumerate(cameras):
            p.camera[:] = [float(c) for c in cam]
            ref.zero_()
            ref8.zero_()
            smax.zero_()
            _abi.check(L.rm_render_device(backend.handle, C.byref(p), ref.data_ptr(), None, smax.data_ptr(), stream))
            _abi.check(L.rm_tonemap_device(C.byref(p), ref.data_ptr(), smax.data_ptr(), 1, ref8.data_ptr(), stream))
            torch.cuda.synchronize()
            same8 = bool(torch.equal(frames8[i], ref8))
            samef = bool(torch.equal(floats[i], ref))
            lit = int((ref8 != 0).any(dim=2).sum())
            detail.append({"camera": list(cam), "rgb8_equal": same8, "float_rows_equal": samef, "nonzero_pixels": lit})
            ok = ok and same8 and samef and lit > 0
            if i == 0:
                sha = hashlib.sha256(frames8[i].cpu().numpy().tobytes()).hexdigest()
    tr.set_camera(cameras[0])
    if world > 1:
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.broadcast(flag, src=0)
        ok = bool(flag.item())
    return ok, sha, detail


def timed_frames(tr, flush, steps, warmup, world, dev):
    """`warmup` untimed frames, then `steps` frames each bracketed by CUDA events on the launching stream, the L2 flushed
    before each (outside its events), barrier + synchronize on both sides; returns (ms per step, max over ranks; the RGB8
    frame of the last step on rank 0, None elsewhere -- valid until the next frame is issued)."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        flush.fill_(1)
        tr.render()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    frame = None
    for a, b in ev:
        flush.fill_(0)
        a.record()
        frame = tr.render()
        b.record()
    barrier()
    if tr.peer is not None:
        tr.peer.status()
    total = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.MAX)
    return float(total[0]) / steps, frame


DUMP_PIXELS = 1 << 20        # pixels kept of a larger frame: 3 x 12 MB of float32 + 8 MB of float64 indices


def dump_outputs(out_dir, tr, frame8):
    """Writes what the last timed step computed, so that two builds can be compared output for output: the RGB8 frame a
    caller receives (frame_rgb8), the float frame it was quantised from (frame_rgb) and the frame's maximum (frame_max).
    A frame of more than DUMP_PIXELS pixels is cut to a fixed sample of pixels drawn with a fixed seed; sample_pixel_index
    holds their flat indices (row * width + column).  Rank 0's buffers only."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    n = tr.height * tr.width
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    sel = torch.from_numpy(idx).to(tr.rgb.device)
    arrays = {"frame_rgb8": frame8.reshape(n, 3)[sel].float(), "frame_rgb": tr.rgb.reshape(n, 3)[sel], "frame_max": tr.dmax}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "sample_pixel_index.npy"), idx.astype(np.float64))


def heavy_leg(name, world, rank, dev, flush, steps=3, warmup=3):
    """The workload that CAN scale (BASELINE.json configs[4] at full size, through the hierarchy) at the same N: a few
    device-timed frames and the same frame check as the headline workload.  Extra key of the bench line; the headline
    (cornell_4k, the metric's configuration) is unchanged."""
    import ctypes as C
    import torch
    import rusty_marcher_b200 as rm
    from rusty_marcher_b200 import _abi, tiled, workloads
    scene_name, w, h, depth, kw, accel = workload_of(name)
    desc = workloads.describe(scene_name, **kw)
    scene = workloads.build_scene(desc)
    r = rm.create_renderer(1.5, h, w)
    r.max_depth, r.accel = depth, accel
    backend = tiled.CudaBackend(scene, r, w, h, dev)
    tr = tiled.TiledRenderer(backend, w, h, dev)
    try:
        L = backend.L
        ms = timed_frames(tr, flush, steps, warmup, world, dev)[0]
        ok, sha, detail = verify_frames(tr, backend, VERIFY_CAMERAS["stress"][:2], world, rank, dev)
        segs = None
        if rank == 0:                                       # segments of the frame: pixels + the queries the kernel counted behind them
            rows = (h // 32) * 32
            q = C.c_uint64(0)
            p = backend.frame_params((0, h // 32))
            scratch = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
            smax = torch.zeros(1, dtype=torch.float32, device=dev)
            _abi.check(L.rm_scene_query_count(backend.handle, C.byref(q), 1))
            _abi.check(L.rm_render_device(backend.handle, C.byref(p), scratch.data_ptr(), None, smax.data_ptr(), torch.cuda.current_stream().cuda_stream))
            _abi.check(L.rm_scene_query_count(backend.handle, C.byref(q), 1))
            segs = rows * w + int(q.value) if accel else None
        return {"workload": name, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms,
                "segments_per_frame": segs, "value": segs / (ms * 1e-3) if segs else None, "unit": UNIT,
                "n_prims": workloads.n_prims(desc), "frame_matches_n1": ok, "frame_sha256": sha, "frame_check": detail,
                "dtype": "f32 (scene queries, shadow rays, lighting) with f64 ray geometry on the reflect / refract paths",
                "timing": "CUDA events around each frame, L2 flushed before each, max over ranks"}
    finally:
        tr.close()
        scene.release()


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import rusty_marcher_b200 as rm
    from rusty_marcher_b200 import _abi, tiled, work, workloads

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world > 1:                           # the library's host threads (delivery of frames): share the box's cores between the ranks
        os.environ.setdefault("RM_B200_HOST_THREADS", str(max(1, (os.cpu_count() or 1) // world)))
    rm.init(local_rank)
    L = _abi.load()

    scene_name, w, h, depth, kw, accel = workload_of(args.workload)
    desc = workloads.describe(scene_name, **kw)
    scene = workloads.build_scene(desc)
    renderer = rm.create_renderer(1.5, h, w)
    renderer.max_depth = depth
    renderer.cull_backfacing = not args.no_cull
    renderer.accel = accel
    backend = tiled.CudaBackend(scene, renderer, w, h, dev)
    tr = tiled.TiledRenderer(backend, w, h, dev)
    rows = (h // 32) * 32

    # ---- algorithmic work of one frame: instrumented kernel, outside the timed region (whole frame, rank 0's GPU)
    fb = rm.FrameBuffer.__new__(rm.FrameBuffer)
    fb.width, fb.height = w, h
    p_all = renderer.params(fb, scene, (0, -1))
    st = _abi.RmStats()
    scratch = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
    smax = torch.zeros(1, dtype=torch.float32, device=dev)
    # (the instrumented kernel walks every primitive like the reference; a frame of configs[4]'s size would take minutes)
    instrumented = rows * w * n_prims_of(desc) <= 1e11
    flops = slots = None
    brute_ms = None
    if instrumented:
        _abi.check(L.rm_render_device_stats(backend.handle, C.byref(p_all), scratch.data_ptr(), None, smax.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream, C.byref(st)))
        counters = st.counters()
        segs = work.segments(counters)
        flops, slots = work.algorithmic_work(counters)
    if accel:
        # segments of the frame from the hierarchy kernel itself: rendered pixels (one primary query each) + the queries it
        # counted behind them (rm_scene_query_count); cross-checked against the instrumented count when there is one
        q = C.c_uint64(0)
        _abi.check(L.rm_scene_query_count(backend.handle, C.byref(q), 1))
        smax.zero_()
        _abi.check(L.rm_render_device(backend.handle, C.byref(p_all), scratch.data_ptr(), None, smax.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
        _abi.check(L.rm_scene_query_count(backend.handle, C.byref(q), 1))
        segs_accel = rows * w + int(q.value)
        if instrumented and abs(segs_accel - segs) > 1e-3 * segs:
            raise SystemExit("bench.py: segment count of the hierarchy kernel (%d) disagrees with the instrumented kernel (%d)" % (segs_accel, segs))
        segs = segs_accel
        if not instrumented:
            st.resident_prims = n_prims_of(desc)
        if instrumented and world == 1:
            # the same frame by brute force (accel = 0), once: what the hierarchy saves
            p_bf = renderer.params(fb, scene, (0, -1))
            p_bf.accel = 0
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            smax.zero_()
            e0.record()
            _abi.check(L.rm_render_device(backend.handle, C.byref(p_bf), scratch.data_ptr(), None, smax.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream))
            e1.record()
            torch.cuda.synchronize()
            brute_ms = e0.elapsed_time(e1)
    walk = None
    if accel:
        # the work the hierarchy kernel itself does for this frame: node visits and leaf tests, counted by its counting
        # instantiation (RmParams.accel = 2) once, outside the timed region -- the roofline numerator of accel workloads
        p_cnt = renderer.params(fb, scene, (0, -1))
        p_cnt.accel = 2
        ws = (C.c_uint64 * 3)()
        _abi.check(L.rm_scene_walk_stats(backend.handle, ws, 1))
        smax.zero_()
        _abi.check(L.rm_render_device(backend.handle, C.byref(p_cnt), scratch.data_ptr(), None, smax.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
        _abi.check(L.rm_scene_walk_stats(backend.handle, ws, 1))
        walk = {"node_visits": int(ws[0]), "sphere_tests": int(ws[1]), "plane_tests": int(ws[2])}
        # per node visit: two slab tests = 2 x (6 sub + 6 mul + 5 min/max + ordering) ~ 50 flop, 64 bytes; leaf tests with
        # SURVEY.md 8d's reject-stage weights (sphere 15, plane 5 + 9 + 6: d.n, distance, point; edge terms not counted);
        # primary ray generation 22 per pixel.  Shading arithmetic is NOT included: a lower bound of the frame's work.
        walk["flops"] = 50 * walk["node_visits"] + 15 * walk["sphere_tests"] + 20 * walk["plane_tests"] + 22 * rows * w
        walk["node_bytes"] = 64 * walk["node_visits"]
        walk["definition"] = ("50 flop + 64 B per node visit (two slab tests), 15 per sphere test, 20 per plane test (SURVEY.md 8d reject-stage "
                              "weights), 22 per primary ray; shading not counted -- a lower bound")
    del scratch

    # ---- FP32 FMA peak, measured live (roofline denominator)
    peak_t, peak_ms = C.c_double(0), C.c_double(0)
    _abi.check(L.rm_measure_fp32_peak(C.byref(peak_t), C.byref(peak_ms)))

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons: nvidia-smi needs ~100 ms to come up and the device-timed region is a few tens of ms, so
    # the sampler runs from here -- warm-up, device-timed region, end-to-end region -- to the end of the e2e loop
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- the timed region: K frames, each bracketed by CUDA events on the launching stream (a frame is the K0 -> K1 pair and
    # nothing else), L2 flushed before each, barrier + synchronize on both sides, max over ranks
    graphs_before = int(L.rm_graph_launch_count())
    ms_per_step, last_frame = timed_frames(tr, flush, args.steps, max(args.warmup, 3), world, dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr, last_frame)
    value = segs / (ms_per_step * 1e-3)
    graphs_headline = int(L.rm_graph_launch_count()) - graphs_before      # frames (warm-up included) issued as one graph launch

    # ---- the same K frames once more with the library's per-kernel events on (K0 | K1 | K4, kept for the last 256 frames):
    # the split of a frame between the kernels.  Not the headline pass: the extra event records between the two launches
    # cost ~5 us per frame (0.0697 against 0.0645 ms on the 4K cornell frame, profiles/r5l_*).
    _abi.check(L.rm_set_profiling(1))
    profiled_ms_per_step = timed_frames(tr, flush, args.steps, 3, world, dev)[0]
    k0_ms, k1_ms, k4_ms = [], [], []
    if tr.exchange == "peer":
        t0, t1, t4 = C.c_double(0), C.c_double(0), C.c_double(0)
        for back in range(min(args.steps, 256)):
            _abi.check(L.rm_kernel_times(back, C.byref(t0), C.byref(t1), C.byref(t4)))
            k0_ms.append(t0.value)
            k1_ms.append(t1.value)
            k4_ms.append(0.0)                # K4 is fused into K1 on this path
    else:                                    # torch.distributed exchange: two library calls per frame, K1 is the first
        t0, t1 = C.c_double(0), C.c_double(0)
        _abi.check(L.rm_last_kernel_times(C.byref(t0), C.byref(t1)))
        k0_ms, k1_ms, k4_ms = [t0.value], [t1.value], [0.0]
    _abi.check(L.rm_set_profiling(0))
    n_k = len(k1_ms)
    total = torch.tensor([sum(k1_ms) / n_k, sum(k0_ms) / n_k, sum(k4_ms) / n_k], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.MAX)
    k1_profiled_ms, k0_ms_avg, k4_ms_avg = (float(x) for x in total)
    # the roofline's kernel duration: the timed region's own events (they bracket the kernel pair of a frame; on the peer
    # path K1 contains the exchange wait and the fused K4)
    k1_ms_avg = ms_per_step if tr.exchange == "peer" else k1_profiled_ms

    # ---- one CUDA graph launch per frame (RM_B200_GRAPH=1, read per call; SURVEY.md 8f row 3) against the two plain launches
    # of the headline, in alternating blocks so that clock drift hits both arms alike
    graph_ab = None
    if os.environ.get("RM_B200_GRAPH") is None:
        n_g = min(args.steps, 100)
        before = int(L.rm_graph_launch_count())
        arms = {"1": [], "0": []}
        for _block in range(3):
            for arm in ("1", "0"):
                os.environ["RM_B200_GRAPH"] = arm
                arms[arm].append(timed_frames(tr, flush, n_g, 3, world, dev)[0])
        del os.environ["RM_B200_GRAPH"]
        graph_ab = {"one_graph_launch_ms_per_frame": sum(arms["1"]) / 3, "two_launches_ms_per_frame": sum(arms["0"]) / 3,
                    "blocks": {"graph": arms["1"], "two_launches": arms["0"]}, "frames_per_block": n_g,
                    "graph_launches": int(L.rm_graph_launch_count()) - before}

    # ---- the frame the ranks assemble against the single-GPU frame: three consecutive frames, the camera moving
    cams = VERIFY_CAMERAS["stress" if scene_name == "stress" else "default"]
    frame_ok, frame_sha, frame_detail = verify_frames(tr, backend, cams, world, rank, dev)
    # the same check with every frame issued as one CUDA graph launch (the first frames of a scene went out as plain
    # launches long ago: all three are graph launches)
    if graph_ab is not None:
        before = int(L.rm_graph_launch_count())
        os.environ["RM_B200_GRAPH"] = "1"
        g_ok, g_sha, _g_detail = verify_frames(tr, backend, cams, world, rank, dev)
        del os.environ["RM_B200_GRAPH"]
        graph_ab["frames_match_n1"] = bool(g_ok and g_sha == frame_sha and int(L.rm_graph_launch_count()) - before == len(cams))
        frame_ok = frame_ok and graph_ab["frames_match_n1"]

    # ---- the workload that can scale, at the same N (extra key; the headline is unchanged)
    heavy = None
    if args.heavy and args.heavy != args.workload:
        heavy = heavy_leg(args.heavy, world, rank, dev, flush)

    # ---- e2e: the public call a user makes -- Renderer.render(frame, scene) with HOST buffers: scene (re)upload H2D and the
    # float frame delivered to host memory inside the timed region.  N = 1: a pinned frame of this process.  N > 1: ONE frame
    # in host memory shared by the ranks (a file in /dev/shm mapped by every process); every rank uploads the scene, renders
    # its bands and delivers them into that frame, timed from a common barrier to the barrier after the last delivery.
    import mmap
    frame = rm.create_frame_buffer(32, 32)
    frame.width, frame.height = w, h
    nbytes = h * w * 12
    pinned, shm_path, shm_map, shm_registered = None, None, None, False
    if world == 1:
        pinned = L.rm_host_alloc(nbytes)
        frame.buffer = (np.ctypeslib.as_array(C.cast(pinned, C.POINTER(C.c_float)), shape=(h, w, 3)) if pinned
                        else np.zeros((h, w, 3), dtype=np.float32))
    else:
        name = [None]
        if rank == 0:
            # shared memory when it has room for the frame (a mapping of a file the tmpfs cannot back dies with SIGBUS on
            # first touch), else a file in the temporary directory: page-cache backed, the same thing to the ranks
            import tempfile
            base = "/dev/shm"
            try:
                st_shm = os.statvfs(base)
                if st_shm.f_bavail * st_shm.f_frsize < nbytes + (64 << 20):
                    base = tempfile.gettempdir()
            except OSError:
                base = tempfile.gettempdir()
            name[0] = os.path.join(base, "rm_b200_bench_%d" % os.getpid())
            with open(name[0], "wb") as f:
                f.truncate(nbytes)
        dist.broadcast_object_list(name, src=0)
        shm_path = name[0]
        fd = os.open(shm_path, os.O_RDWR)
        shm_map = mmap.mmap(fd, nbytes)
        os.close(fd)
        frame.buffer = np.frombuffer(shm_map, dtype=np.float32).reshape(h, w, 3)
        if rank == 0:
            frame.buffer[:] = 7.                 # poisoned: every rendered row must be written by some rank
        barrier()
        # every rank pins its mapping of the shared frame (cudaHostRegister, once, outside the timed region): its device
        # then writes the busy tiles of its bands straight into the frame; a box that refuses keeps the staged delivery
        shm_registered = L.rm_host_register(frame.buffer.ctypes.data, nbytes) == 0
    devnull = open(os.devnull, "w")
    stdout = sys.stdout

    def e2e_loop(fb, n, warm, reupload=True):
        times, d2h_b = [], 0
        for i in range(warm + n):
            flush.fill_(0)
            barrier()
            t0 = time.perf_counter()
            if reupload:
                scene.release()                # force the H2D re-upload of the scene every step
            renderer.render(fb, scene, patch_rows=tr.rows)
            if world > 1:
                dist.barrier()                 # the frame is complete when the last rank has delivered its bands
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
                d2h_b = int(renderer.last_stats.d2h_bytes)
        t = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) * 1e3 / n, d2h_b

    e2e_extra = {}
    try:
        sys.stdout = devnull                   # Renderer.render prints the reference's status lines
        renderer.retained = False
        e2e_ms, d2h = e2e_loop(frame, args.steps, args.warmup)
        n_var = min(args.steps, 50)
        # ... and what a re-render loop that keeps its FrameBuffer pays (main.rs:329-351; RM_ROWS_RETAINED)
        renderer.retained = True
        e2e_extra["retained_ms_per_frame"], e2e_extra["retained_d2h_bytes_per_step"] = e2e_loop(frame, n_var, 5)
        renderer.retained = False
        if world == 1:
            # the reference's own frame type: f64 rows (framebuffer.rs:6-10), pageable memory like a Vec's
            fb64 = rm.create_frame_buffer(w, h, dtype=np.float64)
            e2e_extra["f64_rows_ms_per_frame"], _ = e2e_loop(fb64, n_var, 5)
            renderer.retained = True
            e2e_extra["f64_rows_retained_ms_per_frame"], _ = e2e_loop(fb64, n_var, 5)
            renderer.retained = False
            del fb64
    finally:
        sys.stdout = stdout
    clocks = sampler.stop() if rank == 0 else None
    # the assembled host frame against the frame one GPU delivers (outside the timed region)
    e2e_ok = True
    if rank == 0:
        check = np.zeros((h, w, 3), dtype=np.float32)
        st1 = _abi.RmStats()
        _abi.check(L.rm_render(scene.device_handle(), C.byref(p_all), check.ctypes.data, None, None, C.byref(st1)))
        e2e_ok = bool(np.array_equal(check[:rows], frame.buffer[:rows]))
        del check
    flat = scene.flatten()
    flat_bytes = (C.sizeof(_abi.RmSphere) * flat.c.n_spheres + C.sizeof(_abi.RmPolygon) * flat.c.n_polygons
                  + 24 * flat.c.n_polygon_vertices + (C.sizeof(_abi.RmTriangle) + C.sizeof(_abi.RmReflectance)) * flat.c.n_triangles
                  + C.sizeof(_abi.RmLight) * flat.c.n_lights + C.sizeof(_abi.RmParams))
    # the same call when the caller only wants what main.rs shows or saves: render + normalize + to_vec, the 8-bit frame
    # (24.9 MB over PCIe); extra information next to the headline e2e figure (single GPU only)
    rgb8_ms = None
    if world == 1:
        nb8 = h * w * 3
        pin8 = L.rm_host_alloc(nb8)
        if pin8:
            st8 = _abi.RmStats()
            t8 = []
            for i in range(5 + min(args.steps, 50)):
                flush.fill_(0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _abi.check(L.rm_render(scene.device_handle(), C.byref(p_all), None, None, pin8, C.byref(st8)))
                if i >= 5:
                    t8.append(time.perf_counter() - t0)
            rgb8_ms = 1e3 * sum(t8) / len(t8)
            L.rm_host_free(pin8)
    d2h_t = torch.tensor([d2h], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(d2h_t, op=dist.ReduceOp.SUM)
    d2h = int(d2h_t[0])

    line = None
    if rank == 0:
        # K1 of the slowest rank's share: with N ranks each kernel processes ~1/N of the frame's work
        # (accel workloads: flops / slots are the algorithmic work of the reference's brute-force traversal, SURVEY.md 8d,
        # most of which the hierarchy skips -- the fractions then say how much faster than a perfect brute-force kernel the
        # frame is, not how busy the FP32 pipes are; null when the frame is too large for the instrumented kernel)
        ach_tflops = flops / world / (k1_ms_avg * 1e-3) / 1e12 if flops is not None else None
        issue_frac = (slots / world / (k1_ms_avg * 1e-3)) / (peak_t.value * 1e12 / 2.0) if slots is not None else None
        brute_frac = ach_tflops / peak_t.value if ach_tflops is not None else None
        if walk is not None:
            # accel workloads: the fraction is quoted on the work the hierarchy kernel executes (its own counters), not on
            # the brute-force traversal it replaces (kept as brute_force_equivalent_frac: how far beyond a perfect
            # brute-force kernel the frame is)
            ach_tflops = walk["flops"] / world / (k1_ms_avg * 1e-3) / 1e12
            walk["node_gbs"] = walk["node_bytes"] / world / (k1_ms_avg * 1e-3) / 1e9
            issue_frac = None
        # DRAM bytes of the dominant kernel per launch, from the committed ncu --set full capture of the same workload
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f).get(args.workload)
            if tj and world == 1:
                traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
        except (OSError, ValueError, KeyError):
            pass
        # the HBM view of the same kernel (it is not the bound): driver-measured copy bandwidth of this pool's B200s
        hbm_peak, hbm_src = 6538.9, "fallback: MEASURED_PEAKS.json absent; the figure the driver measured on this pool (torch copy, 2026-10-18)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak, hbm_src = float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json:hbm_gbs"
        except (OSError, ValueError, KeyError):
            pass
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            full_s, threads, sample = cpu_reference_frame_time(desc, w, h, depth, budget_s=25.0, reps=3)
            cpu = {"value": segs / full_s, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                   "ms_per_frame": full_s * 1e3}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_of(args, {
                "segments_per_frame": segs, "pixels_per_frame": rows * w, "resident_prims": st.resident_prims,
                "cull_backfacing": bool(renderer.cull_backfacing),
                "step": ("K0 per-frame records + tile schedule; K1 render + channel max + (fused K4) normalise+quantise of the busy tiles to RGB8"
                         + ("" if world == 1 else ", the exchange inside K1 over NVLink peer memory: max of one float per rank, RGB8 tiles stored straight into rank 0's frame"))
                        if tr.exchange == "peer" else "K0, K1 render + fused max, max all-reduce (NCCL), K4 normalise+quantise RGB8, RGB8 gather to rank 0 (NCCL)",
                "exchange": tr.exchange,
                "frames_as_one_graph_launch": graphs_headline,
                "parallelism": "32-row bands dealt round-robin to %d rank%s" % (world, "" if world == 1 else "s"),
                "l2": "flushed between steps (256 MiB fill, outside each step's CUDA events)"}),
            "ms_per_frame": ms_per_step,
            "frame_matches_n1": frame_ok, "frame_sha256": frame_sha, "frame_check": frame_detail,
            "heavy": heavy,
            "graph_ab": graph_ab,
            "clocks": clocks,
            "e2e": {"value": segs / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_frame": e2e_ms,
                    "h2d_bytes_per_step": flat_bytes * world, "d2h_bytes_per_step": d2h,
                    "path": ("Renderer.render(frame, scene) -> rm_scene_upload + rm_render: float32 frame delivered into pinned host memory -- "
                             "the device writes the busy tiles straight into the frame over PCIe while host threads clear the black tiles"
                             if world == 1 else
                             "every rank: Renderer.render(frame, scene, patch_rows = its bands) -> rm_scene_upload + rm_render into ONE float32 "
                             "frame in host memory shared by the ranks (a mapped file in /dev/shm%s); timed barrier to barrier, max over ranks" % (", pinned by every rank with cudaHostRegister" if shm_registered else "")),
                    "frame_matches_n1": e2e_ok,
                    "pcie_gbs": d2h / (e2e_ms * 1e-3) / 1e9,
                    "host_threads_per_rank": int(os.environ.get("RM_B200_HOST_THREADS", "0")) or os.cpu_count(),
                    "rgb8_only_ms_per_frame": rgb8_ms, **e2e_extra},
            "gpu_launches": tr.launches_per_frame() * args.steps,
            "roofline": {"bound": "fp32", "achieved": ach_tflops, "peak": peak_t.value, "unit": "TFLOP/s",
                         "frac": ach_tflops / peak_t.value if ach_tflops is not None else None, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "render_fast_kernel<false, 1, *> (hierarchy walk)" if accel else "render_fast_kernel<true, 0, *>", "kernel_ms": k1_ms_avg,
                         "kernel_ms_source": "the timed region's CUDA events (each step is the K0 -> K1 pair and nothing else)" if tr.exchange == "peer" else "the library's events around K1",
                         "profiled_pass": {"ms_per_step": profiled_ms_per_step, "k0_plus_k1_ms": k1_profiled_ms,
                                           "note": "second pass of the same frames with the library's per-kernel events on; they cost the difference to ms_per_step"},
                         "work_definition": (walk["definition"] if walk is not None else "reference traversal, resident primitives (SURVEY.md 8d)"),
                         "walk": walk, "brute_force_equivalent_frac": brute_frac if accel else None,
                         "brute_force_ms_same_frame": brute_ms,
                         "prepare_kernel_ms": k0_ms_avg,
                         "kernel_includes": "K0 (prepare) + K1: render + exchange wait + fused K4, CUDA events around both launches" if tr.exchange == "peer" else "render only",
                         "algorithmic_flops_per_frame": flops, "algorithmic_issue_slots_per_frame": slots,
                         "issue_slot_frac": issue_frac,
                         "peak_source": "measured live: ffma_probe_kernel (pure dependent-chain FFMA, all SMs); nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4",
                         "hbm_gbs_achieved": (rows * w * 15 / world) / (k1_ms_avg * 1e-3) / 1e9,
                         "hbm_gbs_peak": hbm_peak, "hbm_peak_source": hbm_src,
                         "hbm_frac": (rows * w * 15 / world) / (k1_ms_avg * 1e-3) / 1e9 / hbm_peak,
                         "hbm_bytes": "12 B/px float rows + 3 B/px RGB8 stored by this kernel (algorithmic)"},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if shm_registered:
        L.rm_host_unregister(frame.buffer.ctypes.data)
    frame.buffer = None
    if pinned:
        L.rm_host_free(pinned)
    if shm_map is not None:
        try:
            shm_map.close()
        except BufferError:
            pass
        if world > 1:
            dist.barrier()
        if rank == 0:
            os.unlink(shm_path)
    tr.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not frame_ok or not e2e_ok or (heavy is not None and not heavy["frame_matches_n1"]):
        sys.stderr.write("bench.py: the frame assembled by %d rank(s) differs from the single-GPU frame\n" % world)
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cornell_4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cull", action="store_true", help="trace every primitive like the reference's brute force")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--heavy", default="stress_8k_bvh", help="second, short leg on a workload that can scale ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float arrays; a seeded pixel sample of a large frame)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
