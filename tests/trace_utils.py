"""Shared helpers for parity tests: seeded synthetic inputs, GPU roll-outs
through the C ABI, golden fixture I/O."""
from __future__ import annotations

import hashlib
import os
from typing import Dict

import numpy as np

from sims import SIMS, make_executor

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make_inputs(sim: str, num_worlds: int, num_steps: int, seed: int = 0) -> Dict[str, np.ndarray]:
    rng = np.random.default_rng(seed)
    if sim == "cartpole":
        return {
            "reset": (rng.random((num_steps, num_worlds, 1)) < 0.01).astype(np.int32),
            "action": rng.integers(0, 2, size=(num_steps, num_worlds, 1), dtype=np.int32),
        }
    if sim == "gridworld":
        return {
            "reset": (rng.random((num_steps, num_worlds, 1)) < 0.02).astype(np.int32),
            "action": rng.integers(0, 5, size=(num_steps, num_worlds, 2), dtype=np.int32),
        }
    if sim in ("room", "room_tgs"):
        # mostly "full speed ahead" so agents reach cubes, walls and each other
        amount = np.where(rng.random((num_steps, num_worlds, 2)) < 0.7, 3,
                          rng.integers(0, 4, size=(num_steps, num_worlds, 2)))
        angle = np.where(rng.random((num_steps, num_worlds, 2)) < 0.7, 0,
                         rng.integers(0, 8, size=(num_steps, num_worlds, 2)))
        act = np.stack([amount, angle,
                        rng.integers(0, 5, size=(num_steps, num_worlds, 2))], axis=-1)
        return {
            "reset": (rng.random((num_steps, num_worlds, 1)) < 0.005).astype(np.int32),
            "action": act.astype(np.int32),
        }
    if sim == "arena":
        shape = (num_steps, num_worlds, 6)
        amount = np.where(rng.random(shape) < 0.6, 3, rng.integers(0, 4, size=shape))
        angle = np.where(rng.random(shape) < 0.6, 0, rng.integers(0, 8, size=shape))
        act = np.stack([amount, angle, rng.integers(0, 5, size=shape),
                        (rng.random(shape) < 0.15).astype(np.int64)], axis=-1)
        return {
            "reset": (rng.random((num_steps, num_worlds, 1)) < 0.004).astype(np.int32),
            "action": act.astype(np.int32),
        }
    if sim in ("balls", "balls_many"):
        return {}          # physics only: no inputs
    raise KeyError(sim)


def rollout_gpu(sim: str, num_worlds: int, num_steps: int, inputs, cfg=None, gpu_id: int = 0):
    """Roll a fixture sim on the B200 engine; returns outputs[name][steps+1, W, ...]."""
    import torch

    desc = SIMS[sim]
    ex = make_executor(sim, num_worlds, gpu_id=gpu_id, **(cfg or {}))
    graph = ex.buildLaunchGraphAllTaskGraphs()
    in_t = {s.name: ex.tensor(s.slot, s.dtype, (num_worlds,) + s.per_world) for s in desc.inputs}
    out_t = {s.name: ex.tensor(s.slot, s.dtype, (num_worlds,) + s.per_world)
             for s in desc.outputs if not s.dynamic}

    def grab(frames):
        for s in desc.outputs:
            if s.dynamic:
                rows = ex.exportedNumRows(s.slot)
                t = ex.tensor(s.slot, s.dtype, (max(rows, 1),) + s.per_world)
                frames[s.name].append(t.cpu().numpy()[:rows].copy())
            else:
                frames[s.name].append(out_t[s.name].cpu().numpy().copy())

    frames = {s.name: [] for s in desc.outputs}
    grab(frames)
    for step in range(num_steps):
        if inputs is not None:
            for s in desc.inputs:
                in_t[s.name].copy_(torch.from_numpy(np.ascontiguousarray(inputs[s.name][step])))
            torch.cuda.synchronize()
        ex.run(graph)
        grab(frames)
    n_kernels = graph.num_kernels
    del graph
    ex.close()
    dyn = {s.name for s in desc.outputs if s.dynamic}
    return {k: (v if k in dyn else np.stack(v)) for k, v in frames.items()}, n_kernels


def save_golden(name, inputs, outs, W, steps):
    payload = {"in_" + k: v for k, v in inputs.items()}
    for k, v in outs.items():
        if isinstance(v, list):
            payload["dyn_" + k] = np.concatenate(v) if v else np.zeros((0,))
            payload["dynlen_" + k] = np.array([len(f) for f in v], dtype=np.int64)
        else:
            payload["out_" + k] = v
    payload["meta"] = np.array([W, steps], dtype=np.int64)
    np.savez_compressed(golden_path(name), **payload)


def load_golden(name):
    z = np.load(golden_path(name))
    ins = {k[3:]: z[k] for k in z.files if k.startswith("in_")}
    outs = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
    for k in z.files:
        if k.startswith("dyn_"):
            lens = z["dynlen_" + k[4:]]
            offs = np.concatenate([[0], np.cumsum(lens)])
            outs[k[4:]] = [z[k][offs[i]:offs[i + 1]] for i in range(len(lens))]
    W, steps = (int(v) for v in z["meta"])
    return W, steps, ins, outs


def assert_traces_equal(got, want, exact=True, rtol=1e-4, atol=1e-6):
    for k, w in want.items():
        g = got[k]
        if isinstance(w, list):
            assert len(g) == len(w), k
            for t, (gf, wf) in enumerate(zip(g, w)):
                assert gf.shape == wf.shape, f"{k} frame {t}: rows {gf.shape} vs {wf.shape}"
                assert np.array_equal(gf, wf), f"{k} frame {t} differs"
        elif exact or not np.issubdtype(w.dtype, np.floating):
            same = g.view(np.uint8) == w.view(np.uint8) if g.dtype.itemsize == 1 else g == w
            if np.issubdtype(w.dtype, np.floating):
                same = g.view(np.uint32) == w.view(np.uint32)
            assert same.all(), f"{k}: first mismatch at {np.argwhere(~same)[0]}"
        else:
            np.testing.assert_allclose(g, w, rtol=rtol, atol=atol, err_msg=k)


def golden_path(name: str) -> str:
    return os.path.join(GOLDEN_DIR, name + ".npz")


# ---- digest goldens: reference traces too large to store whole ---------------------------
# Each column is kept as the SHA-256 of its whole trace (a bit-exact comparison), each frame
# as a short digest of all columns (where a trace starts to differ), and a few seeded values
# of every tenth frame of the float columns (the 1e-4 comparison of MADRONA_B200_FAST_MATH=1).

SAMPLE_VALUES = 4
SAMPLE_EVERY = 10


def _frames(v):
    return [np.ascontiguousarray(f) for f in v]


def _trace_sha(frames) -> np.ndarray:
    h = hashlib.sha256()
    for f in frames:
        h.update(np.int64(f.shape[0]).tobytes())
        h.update(f.tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def _frame_shas(traces, steps) -> np.ndarray:
    out = np.zeros((steps + 1, 8), dtype=np.uint8)
    for t in range(steps + 1):
        out[t] = _trace_sha([traces[k][t] for k in sorted(traces)])[:8]
    return out


def _sample(frames, seed):
    """SAMPLE_VALUES seeded values of every SAMPLE_EVERY-th frame (dynamic tables: the first ones)."""
    size = min(f.size for f in frames)
    idx = np.random.default_rng(seed).choice(size, size=min(SAMPLE_VALUES, size), replace=False)
    return np.stack([f.reshape(-1)[idx] for f in frames[::SAMPLE_EVERY]]) if size else None


def inputs_digest(inputs) -> np.ndarray:
    h = hashlib.sha256()
    for k in sorted(inputs or {}):
        h.update(k.encode())
        h.update(np.ascontiguousarray(inputs[k]).tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def save_digest_golden(name, inputs, outs, W, steps):
    traces = {k: _frames(v) for k, v in outs.items()}
    payload = {"meta": np.array([W, steps], dtype=np.int64), "in_sha": inputs_digest(inputs),
               "frame_sha": _frame_shas(traces, steps)}
    for i, (k, frames) in enumerate(sorted(traces.items())):
        payload["sha_" + k] = _trace_sha(frames)
        payload["dtype_" + k] = np.array(frames[0].dtype.str)
        smp = _sample(frames, i) if np.issubdtype(frames[0].dtype, np.floating) else None
        if smp is not None:
            payload["smp_" + k] = smp
    np.savez_compressed(golden_path(name), **payload)


def assert_matches_digest_golden(got, name, inputs, exact=True, rtol=1e-4, atol=1e-6):
    """`got` (a trace as rollout_gpu returns it) against the digest golden `name`."""
    z = np.load(golden_path(name))
    W, steps = (int(v) for v in z["meta"])
    assert np.array_equal(inputs_digest(inputs), z["in_sha"]), \
        f"{name}: the inputs differ from the ones the golden trace was made from"
    keys = sorted(f[4:] for f in z.files if f.startswith("sha_"))
    traces = {}
    for i, k in enumerate(keys):
        assert len(got[k]) == steps + 1, (k, len(got[k]))
        traces[k] = [np.asarray(f, dtype=np.dtype(str(z["dtype_" + k]))) for f in _frames(got[k])]
        assert all(f.shape[0] == W for f in traces[k]) or isinstance(got[k], list), k
    differ = [k for k in keys if not np.array_equal(_trace_sha(traces[k]), z["sha_" + k])]
    if exact or not differ:
        if differ:
            t = int(np.argmax((_frame_shas(traces, steps) != z["frame_sha"]).any(axis=1)))
            raise AssertionError(f"{name}: columns {differ} differ from the reference, first in frame {t}")
        return
    for i, k in enumerate(keys):
        floating = "smp_" + k in z.files
        assert floating or k not in differ, f"{k} differs from the reference"
        if floating:
            np.testing.assert_allclose(_sample(traces[k], i), z["smp_" + k], rtol=rtol, atol=atol, err_msg=k)


# ---- known-answer probes (oracle/*_probe.cpp) ----------------------------------------------

def reference_probe_output(probe: str) -> str:
    """What the probe printed built against the reference (tests/golden/<probe>.txt.gz)."""
    import gzip
    with gzip.open(os.path.join(GOLDEN_DIR, probe + ".txt.gz"), "rt") as f:
        return f.read()


def build_engine_probe(target: str, out_dir) -> str:
    """Builds oracle/Makefile's `target` (a probe compiled against the engine's own headers
    only) into out_dir, runs it and returns what it printed."""
    import subprocess
    oracle = os.path.join(os.path.dirname(GOLDEN_DIR), os.pardir, "oracle")
    exe = os.path.join(str(out_dir), target)
    subprocess.run(["make", "-s", "-C", oracle, "OUT=" + str(out_dir), exe], check=True,
                   capture_output=True, text=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout
