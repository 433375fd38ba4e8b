"""bench.py's reference arm (CPU: the oracle port timed on the host cores) prints exactly one JSON line that carries
the contract's keys; under a multi-rank launch only rank 0 prints.  On a GPU: the CUDA arm's --steps and --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, gpus=1):
    env = dict(os.environ)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--shape", "toy",
                          "--cpu-budget", "0.5", "--gpus", str(gpus), "--steps", "4"], capture_output=True, text=True, env=env,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_rows_per_s" and d["unit"] == "train rows/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "eval_value": d["eval"]["value"]}
    assert "workload" in d["config"] and d["data"] == "synthetic" and d["scaling"] == "weak"
    assert d["steps"] == 4


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, gpus=2) == []
    lines = _run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, gpus=2)
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and "B=64" in d["config"]["workload"]       # data-parallel arm: global batch 2 x 32


@pytest.mark.gpu
def test_cuda_arm_times_the_requested_steps_and_dumps_its_outputs(tmp_path):
    """--steps sets the timed steps (the kernels launched in the timed window scale with it); --dump-outputs writes
    the headline's outputs after its last timed step as float32 / float64 .npy files; the same arguments give the same
    inputs, hence the same outputs, and one more step gives other outputs."""
    runs = {}
    for tag, steps in (("a", 7), ("b", 7), ("c", 8)):
        d = os.path.join(str(tmp_path), tag)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--shape", "toy", "--steps", str(steps),
                              "--warmup", "3", "--no-cpu-baseline", "--no-alt", "--num-labels", "0", "--no-breakdown",
                              "--dump-outputs", d], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.strip()]
        assert len(lines) == 1
        line = json.loads(lines[0])
        assert line["steps"] == steps
        assert all(f.endswith(".npy") for f in os.listdir(d))
        arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
        assert {"train_loss", "eval_rank", "eval_n_equal", "state__var__ent_emb"} <= set(arrays)
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        assert np.isfinite(arrays["train_loss"]) and arrays["eval_rank"].shape == (32,) and arrays["eval_rank"].min() >= 1
        runs[tag] = (line, arrays)
    (la, a), (lb, b), (lc, c) = runs["a"], runs["b"], runs["c"]
    assert la["gpu_launches"] > 0 and la["gpu_launches"] == lb["gpu_launches"]
    assert lc["gpu_launches"] * 7 == la["gpu_launches"] * 8
    assert set(a) == set(b) == set(c)
    assert np.array_equal(a["eval_rank"], b["eval_rank"])
    assert abs(float(a["train_loss"]) - float(b["train_loss"])) <= 1e-6 * abs(float(b["train_loss"]))
    assert float(c["train_loss"]) != float(a["train_loss"])
    assert not np.array_equal(c["state__var__ent_emb"], a["state__var__ent_emb"])
