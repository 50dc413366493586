"""bench.py contract checks that run without a GPU: the reference arm (`--impl reference`) prints ONE JSON line with the keys
the driver reads, on the same `config` as the GPU arm would use, and the rank > 0 processes of a torchrun launch stay silent.
On a B200: the files of `--dump-outputs`."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--streams", "2", *args],
                       capture_output=True, text=True, env=env, cwd=str(ROOT), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_line():
    lines = _run()
    assert len(lines) == 1
    b = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e"):
        assert key in b, key
    assert b["impl"] == "reference" and b["metric"] == "tracked frames/sec" and b["unit"] == "frames/s" and b["higher_is_better"] is True
    assert b["value"] > 0 and b["e2e"]["value"] == b["value"] and b["e2e"]["h2d_bytes_per_step"] == 0 and b["e2e"]["d2h_bytes_per_step"] == 0
    cb = b["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == b["value"] and cb["streams_lost"] == 0
    assert cb["one_thread_frames_per_s"] > 0 and abs(sum(cb["stage_share"].values()) - 1.0) < 1e-9
    # the same config dict as the GPU arm builds for this command line (the driver compares the two)
    sys.path.insert(0, str(ROOT))
    import bench
    assert b["config"] == bench.vo_config(2, 10)
    assert "C5" in b["config"]["workload"]


def test_reference_arm_is_silent_on_other_ranks():
    lines = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert lines == []


def test_rejects_zero_steps_and_dumps_outside_the_gpu_path():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"], ["--workload", "extract_match", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, cwd=str(ROOT), timeout=60)
        assert r.returncode == 2 and "error" in r.stderr, (args, r.stderr[-500:])


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    """--dump-outputs writes the timed leg's poses of its last step (here frames 40..49 of each stream: 3 warm-up + 2 timed steps
    of 10 frames) and the per-stream counters; the poses are the streams' ground truth to tracking accuracy."""
    from ygz_slam_b200 import se3, synth
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "3", "--streams", "2", "--no-secondary",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=str(ROOT), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    poses, stats = np.load(tmp_path / "poses.npy"), np.load(tmp_path / "tracking_stats.npy")
    assert poses.dtype == stats.dtype == np.float64 and poses.shape == (2, 10, 3, 4) and stats.shape == (2, 12)
    assert np.all(stats[:, 0] == 0) and np.all(stats[:, 1] > 0)                 # no stream lost, key-frames inserted
    for s in range(2):
        truth = synth.shift_stream(s, 50)[2][40:]
        assert max(np.linalg.norm(se3.se3_log(se3.mul(poses[s, k], se3.inv(truth[k])))) for k in range(10)) < 1e-2
