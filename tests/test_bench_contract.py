"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`: the reference's
own algorithm on the host cores, through the oracle -- one of the two places allowed to execute oracle/) prints ONE JSON
line with the keys the driver reads; the GPU arm refuses to run without a device instead of falling back; the workload
table holds BASELINE.json's configurations at their stated sizes."""
import json
import os
import subprocess
import sys

import pytest

from tests.conftest import ROOT, has_gpu

BENCH = os.path.join(ROOT, "bench.py")


def run(*args, timeout=300):
    return subprocess.run([sys.executable, BENCH] + list(args), capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = run("--impl", "reference", "--workload", "cornell_1080p", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ray_segments_per_s" and d["unit"] == "segments/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("cornell_box 1920x1080") and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    # value = segments of the frame / time of the step
    assert abs(d["value"] - d["config"]["segments_per_frame"] / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "patches" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_gpu_arm_refuses_to_run_without_a_device():
    r = run("--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr + r.stdout
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_frame_as_float_arrays(tmp_path):
    """--dump-outputs DIR: the RGB8 frame of the last timed step, its float frame and maximum, as a seeded pixel sample
    of a frame larger than bench.DUMP_PIXELS, float32 / float64 only, 64 MB at most."""
    import numpy as np
    r = run("--workload", "cornell_1080p", "--steps", "2", "--warmup", "0", "--heavy", "", "--no-cpu-baseline",
            "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr
    names = sorted(os.listdir(tmp_path))
    assert names == ["frame_max.npy", "frame_rgb.npy", "frame_rgb8.npy", "sample_pixel_index.npy"]
    assert sum(os.path.getsize(tmp_path / n) for n in names) <= 64 << 20
    a = {n[:-4]: np.load(tmp_path / n) for n in names}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    idx = a["sample_pixel_index"]
    assert idx.shape == (1 << 20,) and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < 1920 * 1080
    rgb8 = a["frame_rgb8"]
    assert rgb8.shape == a["frame_rgb"].shape == (1 << 20, 3)
    assert np.array_equal(rgb8, np.round(rgb8)) and rgb8.min() >= 0 and 0 < rgb8.max() <= 255
    assert a["frame_max"].shape == (1,) and a["frame_max"][0] > 0


def test_dump_outputs_is_refused_by_the_reference_arm():
    r = run("--impl", "reference", "--dump-outputs", "unused")
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_workload_table_holds_the_baseline_configurations():
    sys.path.insert(0, ROOT)
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert base["metric"] and "configs" in base
    W = bench.WORKLOADS
    # name: (scene, width, height, max_depth, scene kwargs)
    assert W["demo"][:4] == ("demo", 1600, 1280, 3)                                  # configs[0]: the reference's CPU-runnable case
    assert W["cornell_4k"][:4] == ("cornell_box", 3840, 2160, 3)                     # configs[1]: the metric's configuration
    assert W["dodecahedron_4k"][:2] == ("dodecahedron", 3840)
    s8 = W["stress_8k_bvh"]
    assert s8[:4] == ("stress", 7680, 4320, 6) and s8[4]["n_spheres"] == 4096 and 2 * s8[4]["grid"] ** 2 + 4096 >= 100_000   # configs[4]
    ap_default = [l for l in open(BENCH) if "--workload" in l and "default=" in l]
    assert ap_default and '"cornell_4k"' in ap_default[0]
