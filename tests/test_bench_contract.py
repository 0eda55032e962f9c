"""bench.py contract checks: the reference arm prints ONE JSON line with the agreed keys; the argument parser accepts
the documented flags; --dump-outputs writes the outputs of the last timed step (end to end on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "sample" in cb and cb["value"] == d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr and out.stdout == ""


def test_dump_outputs_writes_floats_and_a_seeded_sample_above_the_limit(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    B = 1000
    arrays = {"obs": rng.standard_normal((B, 18)).astype(np.float32), "return": rng.standard_normal(B),
              "terminated": rng.random(B) < 0.5, "trajectory_length": rng.integers(1, 201, B).astype(np.int32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == sorted(k + ".npy" for k in arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "all" / f"{k}.npy")
        assert got.dtype in (np.float32, np.float64) and np.array_equal(got, v), k
    limit = 40_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit_bytes=limit)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= limit
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert 0 < len(idx) < B and (np.diff(idx) > 0).all()
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), v[idx.astype(np.int64)]), k
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")), k


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    B = 16384
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--envs-per-gpu", str(B), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout)
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    got = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(got) == {"obs", "return", "terminated", "truncated", "is_success", "is_collided", "end_effector", "trajectory_length"}
    assert all(v.dtype in (np.float32, np.float64) and len(v) == B for v in got.values())
    assert got["obs"].ndim == 2 and got["end_effector"].shape == (B, 2)
    length = got["trajectory_length"]
    assert ((length >= 1) & (length <= 200)).all() and np.isfinite(got["return"]).all()


def test_ncu_numbers_json_is_what_the_committed_summaries_say():
    """bench.py takes every ncu-derived number (dram bytes, executed instructions, pipe shares) from profiles/ncu_numbers.json;
    that file must be exactly what tools/ncu_to_json.py derives from the committed profiles/*_ncu_summary.txt, and bench.py
    itself must not carry such literals"""
    sys.path.insert(0, ROOT)
    from tools import ncu_to_json
    with open(os.path.join(ROOT, "profiles", "ncu_numbers.json")) as f:
        stored = json.load(f)
    assert stored == json.loads(json.dumps(ncu_to_json.build()))
    assert "rollout_config2" in stored and stored["rollout_config2"]["warp_instructions"] > 0
    assert stored["rollout_config2"]["dram_bytes"] > 0 and stored["trajgen_promp"]["dram_bytes"] > 0
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "NCU_TRAFFIC" not in src and "NCU_WARP_INSTRUCTIONS" not in src and "NCU_PIPES" not in src
