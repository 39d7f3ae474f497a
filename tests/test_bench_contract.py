"""bench.py's output contract on the arm that runs without a GPU (--impl reference: the reference's own CPU code, or the
C restatement where the reference build did not travel): stdout is exactly ONE JSON line with the keys the driver reads,
whatever libraries print meanwhile (file descriptor 1 is pointed at stderr for the run)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_exactly_one_json_line():
    env = dict(os.environ, NCCL_DEBUG="VERSION")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, p.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "scan-matches/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["config"]["workload"] == "cfg2" and d["steps"] == 1 and d["warmup"] == 1


def test_product_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], cwd=ROOT,
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and p.stdout.strip() == "" and "no CUDA device" in p.stderr


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: the CorrelateScan results of the last timed step, float64, one row per match of the batch; --steps
    sets the number of timed steps; the same seeded inputs give the same outputs run after run."""
    import numpy as np
    outs = []
    for run in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "0", "--batch", "16",
                            "--no-k2", "--no-cpu-baseline", "--quick", "--dump-outputs", str(tmp_path / run)],
                           cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads(p.stdout)
        assert d["steps"] == 3 and d["multi_gpu_exact"]["ok"]
        got = {n: np.load(tmp_path / run / f"{n}.npy") for n in ("response", "pose", "covariance", "status", "tie_count")}
        assert all(a.dtype == np.float64 for a in got.values())
        assert got["response"].shape == (16,) and got["pose"].shape == (16, 3) and got["covariance"].shape == (16, 3, 3)
        assert (got["status"] == 0).all() and (got["tie_count"] >= 1).all() and (got["response"] > 0).all()
        outs.append(got)
    assert all(np.array_equal(outs[0][n], outs[1][n]) for n in outs[0])
