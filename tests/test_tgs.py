"""Solver::TGS through the same PhysicsSystem API (SURVEY 8f N3).  The reference's TGS
(src/physics/tgs.cpp:59-304) integrates velocities and positions per substep and leaves
its contact / joint prepare, warm-start and solve systems empty, so bodies fall freely;
the engine reproduces exactly that (sims/room built with -DROOM_TGS=1 on both sides)
bit for bit."""
import numpy as np
import pytest

from oracle import runner
from sims import SIMS
from trace_utils import assert_matches_digest_golden, assert_traces_equal, load_golden, make_inputs, rollout_gpu

CFG = {"episode_len": 30, "seed": 8}


@pytest.mark.skipif(not runner.available("room_tgs"), reason="oracle/_ref not built")
def test_reference_backend_reproduces_golden():
    W, steps, ins, outs = load_golden("room_tgs_w3_s45")
    got, _ = runner.run_reference(SIMS["room_tgs"], W, steps, ins, CFG, workers=1)
    assert_traces_equal(got, outs)


def test_golden_shows_the_reference_tgs_has_no_collision_response():
    W, steps, ins, outs = load_golden("room_tgs_w3_s45")
    # dynamic cubes sink through the ground plane (no contact solve in tgs.cpp) ...
    z = np.array([f[16:31, 2] for f in outs["body_pos"][:29]])
    assert z[28].max() < -3.0 and (np.diff(z, axis=0) <= 1e-6).all()
    # ... and the episode reset at step 30 puts new ones back
    assert outs["body_pos"][31][16:31, 2].min() > 0.5


@pytest.mark.gpu
def test_gpu_matches_golden():
    W, steps, ins, outs = load_golden("room_tgs_w3_s45")
    got, n_kernels = rollout_gpu("room_tgs", W, steps, ins, CFG)
    assert n_kernels > 10
    assert_traces_equal(got, outs)


@pytest.mark.gpu
def test_gpu_matches_live_reference():
    # the reference CPU backend's trace is stored as a digest golden (tests/golden/make_golden.py)
    W, steps = 120, 50
    cfg = {"episode_len": 25, "seed": 300}
    ins = make_inputs("room_tgs", W, steps, seed=6)
    got, _ = rollout_gpu("room_tgs", W, steps, ins, cfg)
    assert_matches_digest_golden(got, "room_tgs_w120_s50_ref", ins)
