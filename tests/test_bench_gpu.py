"""bench.py --dump-outputs on the CUDA path: the files hold what the headline's last timed launch left (the oracle's
rollout of the same seeded games over every launch), and --steps sets the number of timed launches."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_launch(tmp_path):
    import torch
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    G, K, steps, seed = 2048, 64, 2, 0x5EED
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", str(steps), "--warmup", "0", "--games", str(G),
                          "--k-steps", str(K), "--no-extras", "--no-cpu-baseline", "--seed", hex(seed), "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == steps
    z = {n: np.load(tmp_path / (n + ".npy")) for n in ("state", "legal_mask", "counters")}
    assert all(a.dtype == np.float64 for a in z.values()) and not (tmp_path / "game_index.npy").exists()
    # every launch (warm-up and timed) advanced each game by K env steps: the oracle does it in one go
    ref = O.fresh_records(G, 2, 1, 0, seed, 0)
    cnt = O.rollout_random(ref, 2, 1, 0, seed, 0, K * (line["warmup"] + steps), threads=8)
    assert np.array_equal(z["counters"], cnt.astype(np.float64))
    eng = BatchedAzul(G, 2, 1, 0, seed=seed, reset=False)
    eng.state.copy_(torch.from_numpy(z["state"].astype(np.int32)))
    assert np.array_equal(eng.export_records().cpu().numpy(), ref)
    for i in range(0, G, 7):
        assert np.array_equal(z["legal_mask"][:, i].astype(np.uint32), O.Game(2, 1, record=ref[i]).legal_mask()), i
