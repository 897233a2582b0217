"""Sphere fixture (sims/balls: a walled pen, loose cubes, a volley of spheres):
sphere-sphere, sphere-plane and -- through the GJK closest-point query --
sphere-hull contacts, B200 engine vs the reference CPU backend.  Same bar as
tests/test_room.py: every exported column BIT-EXACT (1e-4 only with
MADRONA_B200_FAST_MATH=1).  The reference harness links the reference's
narrowphase.cpp / geo.cpp with -DNDEBUG (oracle/Makefile says why)."""
import os

import numpy as np
import pytest

from oracle import runner
from sims import SIMS
from trace_utils import assert_matches_digest_golden, assert_traces_equal, load_golden, rollout_gpu

EXACT = os.environ.get("MADRONA_B200_FAST_MATH", "0") != "1"
CFG = {"seed": 3}


@pytest.mark.skipif(not runner.available("balls"), reason="oracle/_ref not built")
def test_reference_backend_reproduces_golden():
    W, steps, ins, outs = load_golden("balls_w6_s160")
    got, _ = runner.run_reference(SIMS["balls"], W, steps, ins, CFG, workers=1)
    assert_traces_equal(got, outs)


def test_golden_exercises_the_sphere_pairs():
    W, steps, ins, outs = load_golden("balls_w6_s160")
    pos, vel = outs["body_pos"], outs["body_vel"]
    assert pos.shape == (steps + 1, W, 16, 3)
    assert not np.isnan(pos).any()
    balls = pos[:, :, 8:, :]
    # sphere-plane: balls come to rest on the floor at their radius (0.6)
    resting = np.abs(balls[-1, :, :, 2] - 0.6) < 0.02
    assert resting.sum() >= W * 2
    assert balls[:, :, :, 2].min() > -0.3        # squeezed under a cube at worst, never through the floor
    # sphere-hull: balls thrown at the walls (|x|,|y| = 4 - 0.6 at contact) bounce back:
    # the horizontal velocity of some ball flips sign while it is next to a wall
    near_wall = (np.abs(balls[:-1, :, :, :2]) > 3.3).any(axis=-1)
    flipped = (np.sign(vel[:-1, :, 8:, :2]) * np.sign(vel[1:, :, 8:, :2]) < 0).any(axis=-1)
    assert (near_wall & flipped).sum() >= W
    # cubes get pushed around by the balls (sphere-hull against dynamic hulls)
    cubes = pos[:, :, 5:8, :2]
    assert np.abs(cubes[-1] - cubes[0]).max() > 0.05


@pytest.mark.gpu
def test_gpu_matches_golden():
    W, steps, ins, outs = load_golden("balls_w6_s160")
    got, n_kernels = rollout_gpu("balls", W, steps, ins, CFG)
    assert n_kernels > 10
    assert_traces_equal(got, outs, exact=EXACT, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_gpu_matches_live_reference_many_worlds():
    # the reference CPU backend's trace is stored as a digest golden (tests/golden/make_golden.py)
    W, steps = 400, 150
    cfg = {"seed": 7000}
    got, _ = rollout_gpu("balls", W, steps, {}, cfg)
    assert_matches_digest_golden(got, "balls_w400_s150_ref", {}, exact=EXACT, rtol=1e-4, atol=1e-5)


# ---- build variant with 95 bodies per world (-DBALLS_MANY=1) ---------------------------------
MANY_CFG = {"seed": 9}
# more rows and pairs than the defaults allow for (64 rows, 256 candidates, 128 contacts per world)
MANY_ENV = {"MADRONA_B200_MAX_CANDIDATES_PER_WORLD": "4096", "MADRONA_B200_MAX_CONTACTS_PER_WORLD": "2048",
            "MADRONA_B200_ROWS_PER_WORLD": "128"}


@pytest.mark.skipif(not runner.available("balls_many"), reason="oracle/_ref not built")
def test_many_reference_backend_reproduces_golden():
    W, steps, ins, outs = load_golden("balls_many_w2_s60")
    got, _ = runner.run_reference(SIMS["balls_many"], W, steps, ins, MANY_CFG, workers=1)
    assert_traces_equal(got, outs)


@pytest.mark.gpu
def test_many_gpu_matches_golden(monkeypatch):
    for k, v in MANY_ENV.items():
        monkeypatch.setenv(k, v)
    W, steps, ins, outs = load_golden("balls_many_w2_s60")
    assert outs["body_pos"].shape[2] == 95
    got, _ = rollout_gpu("balls_many", W, steps, ins, MANY_CFG)
    assert_traces_equal(got, outs, exact=EXACT, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_many_gpu_matches_live_reference(monkeypatch):
    for k, v in MANY_ENV.items():
        monkeypatch.setenv(k, v)
    W, steps = 48, 80
    cfg = {"seed": 31000}
    got, _ = rollout_gpu("balls_many", W, steps, {}, cfg)
    assert_matches_digest_golden(got, "balls_many_w48_s80_ref", {}, exact=EXACT, rtol=1e-4, atol=1e-5)
