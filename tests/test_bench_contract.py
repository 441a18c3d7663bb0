"""bench.py contract checks that need no GPU: the reference arm (CPU restatement of the reference
path) prints ONE JSON line with the agreed keys, and the product arm refuses to run without CUDA
(there is no CPU fallback to time by accident)."""
import json
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _run(*args, timeout=300):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, cwd=str(ROOT))


def test_reference_arm_prints_one_contract_line():
    r = _run("--impl", "reference", "--workload", "stories15m", "--steps", "8", "--warmup", "3")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "decode_tokens_per_s" and d["unit"] == "tokens/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 8 and d["warmup"] == 3
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "stories15M" in cb["sample"]
    assert d["config"]["workload"].startswith("stories15M") and d["gpu_launches"] == 0
    assert d["vs_baseline"] is None  # BASELINE.md publishes a number for TinyLlama-1.1B fp32 only


def test_reference_arm_other_ranks_exit_quietly(monkeypatch):
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setenv("WORLD_SIZE", "2")
    r = _run("--impl", "reference", "--gpus", "2", "--workload", "stories15m", "--steps", "4", "--warmup", "3")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run("--workload", "stories15m", "--steps", "4", "--warmup", "3", "--no-cpu-baseline")
    assert r.returncode != 0 and r.stdout.strip() == ""


def test_timed_positions_cover_the_metrics_context():
    """--steps is the number of timed positions, not the context: fewer than 1024 steps are spread
    as equal windows over context 1 -> 1024; 1024 or more run the whole context in one window."""
    sys.path.insert(0, str(ROOT))
    import bench
    assert bench.plan_windows(1024, 1024) == [(0, 1024)]
    for steps in (1, 3, 4, 20, 64, 100, 1000):
        w = bench.plan_windows(steps, 1024)
        assert sum(n for _, n in w) == steps and len(w) <= 16
        assert all(0 <= s and s + n <= 1024 for s, n in w)
        assert all(w[i][0] + w[i][1] <= w[i + 1][0] for i in range(len(w) - 1))  # disjoint, ordered
        if len(w) > 1:
            assert w[0][0] == 0 and w[-1][0] + w[-1][1] == 1024  # from context 1 to context 1024
            mean_pos = sum(s + (n - 1) / 2 for s, n in w) / len(w)
            assert abs(mean_pos - 511.5) < 40
    assert bench.plan_windows(20, 1024) == [(0, 4), (255, 4), (510, 4), (765, 4), (1020, 4)]


def test_default_workload_follows_the_metric():
    sys.path.insert(0, str(ROOT))
    import bench
    assert bench.default_workload(2) == bench.default_workload(8) == "llama2-7b-int8"
    import torch
    if not torch.cuda.is_available():
        assert bench.default_workload(1) == "tinyllama-1.1b"


def test_steps_beyond_the_models_context_are_refused():
    r = _run("--workload", "small", "--steps", "161", "--warmup", "3", "--no-cpu-baseline")
    assert r.returncode != 0 and r.stdout.strip() == "" and "exceeds the context" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_repeat(tmp_path):
    """--dump-outputs DIR: the logits and greedy id of the last timed step, identical from run to run
    (same arguments, same seeded inputs); --steps is the number of timed positions."""
    outs = []
    for i in range(2):
        d = tmp_path / str(i)
        r = _run("--workload", "small", "--steps", "12", "--warmup", "3", "--reps", "1", "--no-exact",
                 "--no-cpu-baseline", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 12
        logits, tok = np.load(d / "logits.npy"), np.load(d / "next_token.npy")
        assert logits.dtype == np.float32 and logits.shape == (4096,)
        assert tok.dtype == np.float64 and tok.shape == (1,) and tok[0] == np.argmax(logits)
        outs.append((logits, tok))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
