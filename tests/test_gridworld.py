"""cfg5-class fixture (pure-ECS grid sim): entity create/destroy, compaction /
world sort every step, per-world queries.  Integer state: Entity IDs (gen+id),
row order of the dynamic Item table, rewards, observations and done flags must
all match the reference CPU backend bit-for-bit."""
import numpy as np
import pytest

from oracle import runner
from sims import SIMS
from trace_utils import assert_matches_digest_golden, assert_traces_equal, load_golden, make_inputs, rollout_gpu

CASES = [
    ("gridworld_w32_s150", {"grid_size": 6, "episode_len": 40, "init_items": 6, "seed": 11}),
    ("gridworld_w5_s400", {"grid_size": 3, "episode_len": 97, "init_items": 20, "seed": 3}),
]


@pytest.mark.skipif(not runner.available("gridworld"), reason="oracle/_ref not built")
@pytest.mark.parametrize("name,cfg", CASES)
def test_reference_backend_reproduces_golden(name, cfg):
    W, steps, ins, outs = load_golden(name)
    got, _ = runner.run_reference(SIMS["gridworld"], W, steps, ins, cfg, workers=1)
    assert_traces_equal(got, outs)


def test_golden_invariants():
    W, steps, ins, outs = load_golden("gridworld_w32_s150")
    for t in range(steps + 1):
        counts = outs["item_count"][t, :, 0]
        assert outs["item_entity"][t].shape[0] == counts.sum()
        # entity ids unique among live items
        ids = outs["item_entity"][t][:, 1]
        assert len(np.unique(ids)) == len(ids)
        # obs.numItems equals the world's live item count for both agents
        assert np.array_equal(outs["obs"][t, :, 0, 2], counts) or t == 0
    assert outs["done"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", CASES)
def test_gpu_matches_golden_bit_exact(name, cfg):
    W, steps, ins, outs = load_golden(name)
    got, n_kernels = rollout_gpu("gridworld", W, steps, ins, cfg)
    assert n_kernels >= 4
    assert_traces_equal(got, outs)


@pytest.mark.gpu
def test_gpu_matches_live_reference_many_worlds():
    # enough worlds for several sort tiles and >1 radix pass (W > 255); the reference CPU
    # backend's trace is stored as a digest golden (tests/golden/make_golden.py)
    W, steps = 3000, 120
    cfg = {"grid_size": 5, "episode_len": 30, "init_items": 10, "seed": 5}
    ins = make_inputs("gridworld", W, steps, seed=77)
    got, _ = rollout_gpu("gridworld", W, steps, ins, cfg)
    assert_matches_digest_golden(got, "gridworld_w3000_s120_ref", ins)
