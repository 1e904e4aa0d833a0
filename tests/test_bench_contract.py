"""bench.py contract on a box without a GPU: the reference arm (the oracle on the host cores) prints one JSON line with the
keys its readers rely on, non-zero ranks of a multi-rank launch stay silent, and the GPU arm refuses to run (no CPU fallback).
On the GPU: --steps sets the timed steps and --dump-outputs writes the frames of the last one."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
SMALL = ["--steps", "1", "--warmup", "1", "--cpu-distinct-frames", "4", "--cpu-frames-per-step", "6"]


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--gpus", "1"] + SMALL)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "stabilized_frames_per_sec_1080p_lk_full_lock" and d["unit"] == "frames/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("c2_lk_full_lock_1080p")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--gpus", "2"] + SMALL, env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)


def test_steps_and_dump_outputs_arguments_are_checked(tmp_path):
    out = tmp_path / "dump"
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(out)] + SMALL,
                 ["--workload", "c5", "--dump-outputs", str(out)]):
        r = _run(args)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-2000:])
    assert not out.exists()


GPU_SMALL = ["--warmup", "2", "--frames-per-gpu", "64", "--batch", "64", "--no-e2e", "--no-cpu-baseline", "--no-c5-probe",
             "--no-parity", "--no-mode-probes"]


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """One and two timed steps over the same seeded clip leave the same frames, the second step's launches are counted in
    the timed region, and the dump is float32 within its budget: the last call complete, every call at the sampled pixels."""
    import bench
    lines, dumps = [], []
    for steps in (1, 2):
        d = tmp_path / f"steps{steps}"
        r = _run(["--steps", str(steps), "--dump-outputs", str(d)] + GPU_SMALL)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0]))
        assert sorted(p.name for p in d.iterdir()) == ["frame_last.npy", "frames_sampled.npy"]
        assert sum(p.stat().st_size for p in d.iterdir()) <= bench.DUMP_BYTES
        dumps.append({p.stem: np.load(p) for p in d.iterdir()})
    assert [l["steps"] for l in lines] == [1, 2]
    assert lines[1]["gpu_launches"] == 2 * lines[0]["gpu_launches"] > 0
    last, sampled = dumps[0]["frame_last"], dumps[0]["frames_sampled"]
    assert last.dtype == sampled.dtype == np.float32
    assert last.shape == (bench.H, bench.W, 3) and sampled.shape == (64, bench.DUMP_PIXELS, 3)
    assert np.array_equal(sampled[-1], last.reshape(-1, 3)[bench.sample_pixels(bench.H, bench.W, bench.DUMP_PIXELS)])
    assert last.std() > 0 and np.array_equal(last, np.clip(np.round(last), 0, 255))
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name]), name
