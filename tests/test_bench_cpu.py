"""bench.py's reference arm (the C oracle port on the host cores) runs without a GPU and prints one JSON line
with the contract's keys."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--k-steps", "64", "--pyref-seconds", "0"], capture_output=True, text=True, timeout=300, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "env_steps/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and line["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--k-steps", "64"], capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_python_reference_leg_when_the_reference_is_staged():
    """cpu_baseline.python_reference: the UNMODIFIED reference's GameRunner loop from baseline/_ref (staged by build());
    reports 'unavailable' instead of failing where the tree was not staged."""
    import pytest
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--k-steps", "64", "--pyref-seconds", "2"], capture_output=True, text=True, timeout=300, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    py = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]["python_reference"]
    if not os.path.isdir(os.path.join(REPO, "baseline", "_ref", "azulnet")):
        assert "unavailable" in py
        pytest.skip("baseline/_ref not staged")
    assert py["kind"] == "reference" and py["cores"] >= 1 and py["games"] > 0 and py["value"] > 100
    assert py["single_core_value"] > 100 and py["unit"] == "env_steps/s" and "cpu_model" in py


def test_dump_outputs_types_budget_and_seeded_sample(tmp_path, monkeypatch):
    """--dump-outputs' writer: integers as float64, floats as float32; over the budget every per-game array keeps the same
    seeded sample of games (game_index.npy), identical from run to run."""
    import numpy as np
    import torch
    import bench
    state = torch.arange(17 * 1000, dtype=torch.int32).reshape(17, 1000) - (1 << 31)
    per_game = {"state": state, "logp": torch.linspace(-1.0, 0.0, 1000)}
    whole = {"counters": torch.arange(16, dtype=torch.int64)}
    bench.dump_outputs(str(tmp_path / "full"), per_game, whole)
    assert sorted(os.listdir(tmp_path / "full")) == ["counters.npy", "logp.npy", "state.npy"]
    assert np.array_equal(np.load(tmp_path / "full" / "state.npy"), state.numpy().astype(np.float64))
    monkeypatch.setattr(bench, "DUMP_BYTES", 40000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), per_game, whole)
    z = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("state", "logp", "counters", "game_index")}
    assert z["state"].dtype == np.float64 and z["logp"].dtype == np.float32 and z["counters"].dtype == np.float64
    assert sum(a.nbytes for a in z.values()) <= 40000
    idx = z["game_index"].astype(np.int64)
    assert 0 < len(idx) < 1000 and np.array_equal(z["state"], state.numpy()[:, idx].astype(np.float64))
    assert np.array_equal(z["logp"], per_game["logp"].numpy()[idx])
    for n in z:
        assert np.array_equal(z[n], np.load(tmp_path / "b" / (n + ".npy")))


def test_dump_outputs_is_refused_for_the_reference_arm():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                         capture_output=True, text=True, timeout=120, cwd=REPO)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
