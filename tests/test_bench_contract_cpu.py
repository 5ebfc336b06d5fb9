"""bench.py contract on CPU: the reference arm (--impl reference = the fp64 oracle port on the host cores) prints ONE JSON line with
the keys the driver reads; ranks other than 0 print nothing."""
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run(extra_env):
    env = dict(os.environ, SMPLSIM_BENCH_SECS="0.3", **extra_env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_json_line():
    lines = _run({"RANK": "0", "WORLD_SIZE": "1"})
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["n_gpus"] == 2
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("cfg2") and d["metric"].startswith("env-steps/sec")


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_dump_outputs_writes_float_arrays_and_samples_envs_above_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.default_rng(1)
    outs = {"obs": rng.normal(size=(50, 7)).astype(np.float32), "reward": rng.random(50).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "all"), outs)
    assert sorted(os.listdir(tmp_path / "all")) == ["obs.npy", "reward.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "obs.npy"), outs["obs"])
    monkeypatch.setattr(bench, "DUMP_BYTES", 20 * (8 * 4 + 8))          # room for 20 of the 50 envs
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    ids = np.load(tmp_path / "a" / "env_ids.npy")
    assert ids.dtype == np.float64 and len(ids) == 20 and np.array_equal(ids, np.load(tmp_path / "b" / "env_ids.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "obs.npy"), outs["obs"][ids.astype(int)])
    assert sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES
