"""BASELINE.json full-size configurations on the GPU, checked through
size-independent properties (the reference CPU backend cannot run these sizes:
its tmp allocator alone is 32 MiB per world).  The reference runs of the first
worlds are stored as digest goldens (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from sims import SIMS
from trace_utils import assert_matches_digest_golden, make_inputs


def _rollout_prefix(sim, W, steps, ins, cfg, keep_worlds, rows_per_world=None):
    """Roll W worlds on the GPU but keep only the first `keep_worlds` worlds."""
    import torch
    from sims import make_executor

    desc = SIMS[sim]
    ex = make_executor(sim, W, **cfg)
    graph = ex.buildLaunchGraphAllTaskGraphs()
    in_t = {s.name: ex.tensor(s.slot, s.dtype, (W,) + s.per_world) for s in desc.inputs}
    out_t = {s.name: ex.tensor(s.slot, s.dtype, (W,) + s.per_world) for s in desc.outputs if not s.dynamic}
    frames = {k: [v[:keep_worlds].cpu().numpy().copy()] for k, v in out_t.items()}
    for step in range(steps):
        for s in desc.inputs:
            full = torch.zeros((W,) + s.per_world, dtype=in_t[s.name].dtype, device=in_t[s.name].device)
            full[:keep_worlds] = torch.from_numpy(np.ascontiguousarray(ins[s.name][step])).to(full.device)
            if s.name == "action" and sim in ("room", "arena"):
                full[keep_worlds:, :, 2] = 2      # neutral turn for the rest
            in_t[s.name].copy_(full)
        torch.cuda.synchronize()
        ex.run(graph)
        for k, v in out_t.items():
            frames[k].append(v[:keep_worlds].cpu().numpy().copy())
    ex.close()
    return {k: np.stack(v) for k, v in frames.items()}


@pytest.mark.gpu
def test_room_8192_worlds_prefix_equals_reference():
    # configs[1]: 8192 worlds / GPU.  Worlds are independent and seeded by their
    # index, so worlds [0, 64) of the 8192-world GPU run must equal a 64-world run
    # of the reference CPU backend -- bit for bit.
    W, keep, steps = 8192, 64, 60
    cfg = {"episode_len": 40, "seed": 7}
    ins = make_inputs("room", keep, steps, seed=31)
    got = _rollout_prefix("room", W, steps, ins, cfg, keep)
    assert_matches_digest_golden(got, "room_w64_s60_prefix_ref", ins)


@pytest.mark.gpu
def test_gridworld_65536_worlds_prefix_equals_reference():
    # configs[4]: 65536 worlds / GPU (3 radix passes, multi-tile onesweep)
    W, keep, steps = 65536, 128, 60
    cfg = {"grid_size": 6, "episode_len": 25, "init_items": 8, "seed": 3}
    ins = make_inputs("gridworld", keep, steps, seed=13)
    got = _rollout_prefix("gridworld", W, steps, ins, cfg, keep)
    assert_matches_digest_golden(got, "gridworld_w128_s60_prefix_ref", ins)


@pytest.mark.gpu
def test_room_8192_worlds_is_deterministic_and_finite():
    W, steps = 8192, 30
    cfg = {"episode_len": 20, "seed": 99}
    ins = make_inputs("room", 8, steps, seed=2)
    a = _rollout_prefix("room", W, steps, ins, cfg, 8)
    b = _rollout_prefix("room", W, steps, ins, cfg, 8)
    for k in a:
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k
        assert np.isfinite(a[k].astype(np.float64)).all()


@pytest.mark.gpu
def test_arena_4096_worlds_prefix_equals_reference():
    # configs[2]: 4096 worlds / GPU.  Worlds [0, 48) of the 4096-world GPU run must equal
    # a 48-world run of the reference CPU backend bit for bit (an episode reset inside).
    W, keep, steps = 4096, 48, 70
    cfg = {"episode_len": 45, "seed": 11}
    ins = make_inputs("arena", keep, steps, seed=77)
    got = _rollout_prefix("arena", W, steps, ins, cfg, keep)
    assert_matches_digest_golden(got, "arena_w48_s70_prefix_ref", ins)
