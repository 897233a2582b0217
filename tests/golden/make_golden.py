"""Generates tests/golden/*.npz by running the fixture simulators on the
*reference* CPU backend (oracle/_ref, built from /root/reference by
oracle/Makefile).  Run where /root/reference exists:

    make -C oracle && python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle.runner import run_reference  # noqa: E402
from sims import SIMS  # noqa: E402
from trace_utils import golden_path, load_golden, make_inputs, save_digest_golden, save_golden  # noqa: E402

CASES = [
    # (file, sim, worlds, steps, cfg)
    ("cartpole_w64_s300", "cartpole", 64, 300, {"max_steps": 200, "seed": 0}),
    ("cartpole_w3_s50", "cartpole", 3, 50, {"max_steps": 10, "seed": 7}),
    ("gridworld_w32_s150", "gridworld", 32, 150,
     {"grid_size": 6, "episode_len": 40, "init_items": 6, "seed": 11}),
    # tiny grid + long episodes: many pickups, item table saturates at kMaxItems
    ("gridworld_w5_s400", "gridworld", 5, 400,
     {"grid_size": 3, "episode_len": 97, "init_items": 20, "seed": 3}),
    # rigid-body room: two resets inside the trace (episode_len 100 + random resets)
    ("room_w4_s210", "room", 4, 210, {"episode_len": 100, "seed": 21}),
    # same fixture with agent 0 grabbing / releasing cubes through fixed joints
    ("room_grab_w3_s120", "room", 3, 120, {"episode_len": 70, "seed": 5, "grab_period": 5}),
    # Hide&Seek-class arena: wedge / hexagonal hulls, latched doors (fixed joints to static
    # walls), grab (fixed) and shove (one-step hinge) joints, two resets inside the trace
    ("arena_w2_s200", "arena", 2, 200, {"episode_len": 90, "seed": 17}),
    # Solver::TGS through the same API (tgs.cpp: integrate velocities / positions only)
    ("room_tgs_w3_s45", "room_tgs", 3, 45, {"episode_len": 30, "seed": 8}),
    # spheres: sphere-sphere, sphere-plane and sphere-hull (GJK) contacts
    ("balls_w6_s160", "balls", 6, 160, {"seed": 3}),
    # 95 bodies per world: candidate search beyond one 64-leaf mask word, ~300 contacts per world
    ("balls_many_w2_s60", "balls_many", 2, 60, {"seed": 9}),
]

# Larger reference runs, stored as digest goldens (trace_utils.save_digest_golden):
# (file, sim, worlds, steps, cfg, input seed (None: no inputs), workers, fixed-size columns only)
DIGEST_CASES = [
    # BASELINE.json configs[0]: 256 worlds, 1000 steps, random actions (tests/test_cartpole.py)
    ("cartpole_w256_s1000_ref", "cartpole", 256, 1000, {}, 42, 1, False),
    # enough worlds for several sort tiles and > 1 radix pass (tests/test_gridworld.py)
    ("gridworld_w3000_s120_ref", "gridworld", 3000, 120,
     {"grid_size": 5, "episode_len": 30, "init_items": 10, "seed": 5}, 77, 8, False),
    # tests/test_room.py
    ("room_w300_s130_ref", "room", 300, 130, {"episode_len": 60, "seed": 1000}, 9, 4, False),
    ("room_grab_w200_s90_ref", "room", 200, 90, {"episode_len": 50, "seed": 77, "grab_period": 3}, 4, 4, False),
    # tests/test_arena.py, tests/test_balls.py, tests/test_tgs.py
    ("arena_w160_s150_ref", "arena", 160, 150, {"episode_len": 60, "seed": 4000}, 21, 4, False),
    ("balls_w400_s150_ref", "balls", 400, 150, {"seed": 7000}, None, 4, False),
    ("balls_many_w48_s80_ref", "balls_many", 48, 80, {"seed": 31000}, None, 4, False),
    ("room_tgs_w120_s50_ref", "room_tgs", 120, 50, {"episode_len": 25, "seed": 300}, 6, 4, False),
    # the first worlds of the BASELINE.json full-size runs (tests/test_full_size.py)
    ("room_w64_s60_prefix_ref", "room", 64, 60, {"episode_len": 40, "seed": 7}, 31, 4, True),
    ("gridworld_w128_s60_prefix_ref", "gridworld", 128, 60,
     {"grid_size": 6, "episode_len": 25, "init_items": 8, "seed": 3}, 13, 4, True),
    ("arena_w48_s70_prefix_ref", "arena", 48, 70, {"episode_len": 45, "seed": 11}, 77, 4, True),
]

if __name__ == "__main__":
    only = sys.argv[1:]
    for name, sim, W, steps, cfg in CASES:
        if only and name not in only:
            continue
        inputs = make_inputs(sim, W, steps, seed=1234)
        outs, _ = run_reference(SIMS[sim], W, steps, inputs, cfg, workers=1)
        save_golden(name, inputs, outs, W, steps)
        print(name, {k: (v.shape if not isinstance(v, list) else f"{len(v)} frames")
                     for k, v in outs.items()})

    # the grab trace's inputs without grabbing: the joints' effect on the bodies
    if not only or "room_nograb_w3_s120" in only:
        W, steps, inputs, _ = load_golden("room_grab_w3_s120")
        outs, _ = run_reference(SIMS["room"], W, steps, inputs, {"episode_len": 70, "seed": 5}, workers=1)
        np.savez_compressed(golden_path("room_nograb_w3_s120"), body_pos=np.stack(outs["body_pos"][::10]))
        print("room_nograb_w3_s120 (body_pos of every tenth frame)")

    for name, sim, W, steps, cfg, seed, workers, fixed_only in DIGEST_CASES:
        if only and name not in only:
            continue
        inputs = {} if seed is None else make_inputs(sim, W, steps, seed=seed)
        outs, _ = run_reference(SIMS[sim], W, steps, inputs, cfg, workers=workers)
        if fixed_only:
            outs = {k: v for k, v in outs.items() if not isinstance(v, list)}
        save_digest_golden(name, inputs, outs, W, steps)
        print(name, sorted(outs))

    # the reference's physics asset pipeline on the hulls of tests/test_physics_assets.py
    if not only or "assets_probe_ref" in only:
        import hashlib
        import subprocess
        import tempfile
        from test_physics_assets import _case, _write_probe_input
        with tempfile.TemporaryDirectory() as tmp:
            inp, outp = os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.bin")
            _write_probe_input(inp, *_case())
            subprocess.run([os.path.join(ROOT, "oracle", "_ref", "assets_probe_ref"), inp, outp],
                           check=True, timeout=120)
            np.savez_compressed(os.path.join(ROOT, "tests", "golden", "assets_probe_ref.npz"),
                                input_sha256=hashlib.sha256(open(inp, "rb").read()).hexdigest(),
                                output=np.fromfile(outp, dtype=np.uint8))
        print("assets_probe_ref")

    # the known-answer probe built against the reference headers: its whole output; the GJK
    # probe: its known answers (the rest is pinned by gjk_probe.sha256)
    for probe in ("kat_probe_ref", "gjk_probe_ref"):
        if only and probe not in only:
            continue
        import gzip
        import subprocess
        text = subprocess.run([os.path.join(ROOT, "oracle", "_ref", probe)],
                              capture_output=True, text=True, check=True).stdout
        if probe == "gjk_probe_ref":
            text = "".join(ln for ln in text.splitlines(keepends=True) if ln.startswith("kat_"))
        with gzip.GzipFile(os.path.join(ROOT, "tests", "golden", probe + ".txt.gz"), "wb", mtime=0) as f:
            f.write(text.encode())
        print(probe, len(text.splitlines()), "lines")

    # digest of the reference GJK probe (oracle/gjk_probe.cpp built against the
    # reference's src/physics/gjk.hpp + geo.cpp): lets the engine's header be
    # checked where oracle/_ref/gjk_probe_ref is absent
    if not only or "gjk_probe" in only:
        import hashlib
        import subprocess
        probe = os.path.join(ROOT, "oracle", "_ref", "gjk_probe_ref")
        text = subprocess.run([probe], capture_output=True, text=True, check=True).stdout
        with open(os.path.join(ROOT, "tests", "golden", "gjk_probe.sha256"), "w") as f:
            f.write(hashlib.sha256(text.encode()).hexdigest() + "\n")
        print("gjk_probe", len(text.splitlines()), "values")
