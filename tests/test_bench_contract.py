"""bench.py contract: the reference arm runs without a GPU and prints one JSON line with the required keys; on a GPU,
--dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["value"] > 1.0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    import torch

    import pqmf_b200 as pq

    dump = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-other-configs",
                        "--dump-outputs", str(dump)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    assert sorted(os.listdir(dump)) == ["reconstruction.npy", "subbands.npy"]
    sub, rec = np.load(dump / "subbands.npy"), np.load(dump / "reconstruction.npy")
    assert sub.dtype == np.float32 and rec.dtype == np.float32
    assert sub.shape == (4, 16, 1 << 16) and rec.shape == (4, 1, 1 << 20)
    assert sub.nbytes + rec.nbytes <= 64 << 20
    # the two files are the forward and the inverse of the same step (a 4-row batch may take another kernel family: tolerance)
    again = pq.PQMF(100, 16).cuda().inverse(torch.from_numpy(sub).cuda()).cpu().numpy()
    assert np.abs(again - rec).max() <= 1e-5
