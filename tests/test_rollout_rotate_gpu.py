"""The rotating rollout kernel (`k_rollout_rotate`: 32-game batches handed round the warps of a block, idle warps asleep on
an mbarrier until a batch is parked in their slot or the block's last batch has finished) at the sizes where the library
chooses it, against the non-rotating kernel and the C oracle.  Needs a B200: run with ``-m gpu``."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from bench import rollout_kernel_name  # noqa: E402
from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


def engine(*a, **k):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    return BatchedAzul(*a, **k)


def kernel(n, players, pool):
    return rollout_kernel_name(n, players, pool, torch.cuda.get_device_properties(0).multi_processor_count, False)


def rollout(eng, k):
    mask = torch.zeros((6, eng.n_games), dtype=torch.int32, device=eng.device)
    eng.rollout_random(k, mask_out=mask)
    return mask


@pytest.mark.parametrize("players,pool", [(2, 1), (3, 0), (4, 1)])
def test_long_rotating_launch_matches_non_rotating_halves(players, pool):
    """65,536 games x 4,096 steps in one launch: about 12 hand-overs per batch, the termination of every block, and a last
    block of 4 batches on 16 warps.  The two 32,768-game halves run the non-rotating kernel (7 warps per block)."""
    n, k, seed, h = 65536, 4096, 0x5EED, 32768
    assert kernel(n, players, pool).startswith("k_rollout_rotate") and kernel(h, players, pool).startswith("k_rollout_random")
    one = engine(n, players, pool, 0, seed=seed)
    m1 = rollout(one, k)
    lo = engine(h, players, pool, 0, seed=seed, game_id_base=0)
    hi = engine(h, players, pool, 0, seed=seed, game_id_base=h)
    m_lo, m_hi = rollout(lo, k), rollout(hi, k)
    assert torch.equal(one.state[:, :h], lo.state) and torch.equal(one.state[:, h:], hi.state)
    assert torch.equal(m1[:, :h], m_lo) and torch.equal(m1[:, h:], m_hi)
    assert torch.equal(one.counters, lo.counters + hi.counters)
    assert int(one.counters[0]) == n * k and int(one.counters[1]) > 0


@pytest.mark.parametrize("k", [3, 700])
def test_small_rotating_blocks_match_oracle(k):
    """9,000 games: blocks of 2 batches + 2 idle warps, the last block with one full and one 8-game batch.  k = 3 ends every
    batch before its first end-of-round pass (no hand-over); k = 700 hands batches over and ends them in every block."""
    players, pool, seed, n, gid0 = 3, 1, 777, 9000, 11
    assert kernel(n, players, pool).startswith("k_rollout_rotate")
    ref = O.fresh_records(n, players, pool, 0, seed, gid0)
    cref = O.rollout_random(ref, players, pool, 0, seed, gid0, k, threads=8)
    eng = engine(n, players, pool, 0, seed=seed, game_id_base=gid0)
    rollout(eng, k)
    assert np.array_equal(eng.export_records().cpu().numpy(), ref)
    assert np.array_equal(eng.counters.cpu().numpy(), cref)
