"""CPU: the reference arm of bench.py runs here (it times the oracle port, no GPU) and prints ONE JSON line with the
keys the driver reads; the roofline arithmetic of the main arm is the one SURVEY.md §8d / DESIGN.md §5 state."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "UAV env-steps/sec" and d["unit"] == "UAV env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 3 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_algorithmic_bytes_follow_the_survey():
    sys.path.insert(0, ROOT)
    import bench

    assert bench.algorithmic_bytes_per_unit("multi", 8) == 110.0       # 41 read + 66 written + 24/N counters
    assert bench.algorithmic_bytes_per_unit("multi", 32) == 107.75
    assert bench.algorithmic_bytes_per_unit("single", 1) == 89.0
    assert set(bench.WORKLOADS) == {"c1", "c2", "c3", "c4", "c4s", "c5", "c5r"}
    assert bench.WORKLOADS["c3"]["B"] == 65536 and bench.WORKLOADS["c3"]["N"] == 8
    assert bench.WORKLOADS["c4s"]["B"] == 1048576 and bench.WORKLOADS["c4s"]["N"] == 32 and bench.WORKLOADS["c4s"]["shard_total"]


def test_reference_arm_runs_the_full_batch_and_the_literal_reference():
    """Same config as the GPU arm (BASELINE configs[2]: all 65,536 envs per step) and, where the literal reference is
    reachable (/root/reference here, oracle/_ref on the GPU box), its single-core number beside the port's."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["config"]["envs_per_step"] == 65536 and d["config"]["envs_per_gpu"] == 65536 and d["config"]["uavs_per_env"] == 8
    lit = d["cpu_baseline_literal"]
    assert "unavailable" in lit or (lit["kind"] == "reference" and lit["cores"] == 1 and 1e3 < lit["value"] < d["value"])


def test_multi_gpu_default_workload_is_configs3():
    """`--gpus N>1` with no --workload measures BASELINE configs[3]: N=32, 1,048,576 envs in total, sharded."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["config"]["uavs_per_env"] == 32 and d["config"]["envs_total"] == 1048576 and d["config"]["envs_per_gpu"] == 131072
    assert d["scaling"] == "strong"


def test_output_sample_keeps_the_same_envs_of_every_array_within_the_budget(monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    import torch

    gen = torch.Generator().manual_seed(0)
    arrays = dict(obs=torch.rand((1000, 8, 10), generator=gen), reward=torch.rand((1000, 8), generator=gen, dtype=torch.float64),
                  done=torch.randint(0, 2, (1000, 8), generator=gen, dtype=torch.uint8))
    whole = bench.output_sample(arrays)
    assert np.array_equal(whole["env_index"], np.arange(1000)) and whole["done"].dtype == np.float32
    assert whole["reward"].dtype == np.float64 and np.array_equal(whole["obs"], arrays["obs"].numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (8 + 8 * 10 * 4 + 8 * 8 + 8 * 4))
    a, b = bench.output_sample(arrays), bench.output_sample(arrays)
    idx = a["env_index"].astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and all(np.array_equal(a[k], b[k]) for k in a)
    for k, v in arrays.items():
        assert np.array_equal(a[k], v.numpy()[idx])


def test_bench_rejects_steps_it_would_not_time():
    for extra in (["--steps", "0"], ["--workload", "c5r", "--steps", "3"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                             cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr and out.stdout == ""


@pytest.mark.gpu
@pytest.mark.parametrize("headline", ["rollout", "per_step"])
def test_dump_outputs_repeat_and_follow_steps(tmp_path, headline):
    """Two runs with the same arguments write the same arrays; a different --steps writes different ones."""

    def run(steps, name):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                              "--no-acting", "--headline", headline, "--dump-outputs", str(tmp_path / name)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        files = sorted(os.listdir(tmp_path / name))
        assert files == ["done.npy", "env_index.npy", "obs.npy", "reward.npy"]
        return {f[:-4]: np.load(tmp_path / name / f) for f in files}

    a, b, c = run(3, "a"), run(3, "b"), run(5, "c")
    assert a["obs"].shape == (65536, 8, 10) and a["obs"].dtype == np.float32
    assert sum(v.nbytes for v in a.values()) <= 64e6
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["obs"], c["obs"])
