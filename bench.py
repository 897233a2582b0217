#!/usr/bin/env python
"""bench.py -- aggregate env-steps/s of the batched ECS step engine.

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference]
                    [--dump-outputs DIR]

A "step" = one pass of the simulator's step task graph over all worlds
(MWCudaExecutor::run equivalent).  One process per GPU (torchrun for N>1);
worlds shard across ranks with no data-path collective, the only exchange is
the gather of the exported reward/done tensors after each step (SURVEY.md 8e):
one NVLink peer-store kernel per rank per step into every peer's symmetric
buffer (madrona_b200/csrc/peer_gather.cu), consumed one step later so it
overlaps the next step graph; `--gather nccl` selects ONE packed
all_gather_into_tensor per step on a side stream instead.  Prints ONE JSON
line on rank 0.

  value     device-timed throughput with inputs already resident in HBM:
            K steps, each bracketed by CUDA events on the launching stream;
            the time is the SUM of the per-step intervals (the 256 MiB L2 flush
            between steps is excluded), max over ranks.  `run_loop` next to it
            is the plain wall clock of K back-to-back run() calls (no flush).
  e2e       same metric through the C ABI with HOST buffers: every step copies
            the actions H2D from pinned memory and reads rewards+dones back D2H.
  roofline  dominant node of the step (per-node CUDA-event timing inside this
            process via mb2_profile_nodes) vs MEASURED_PEAKS.json hbm_gbs.
  --dump-outputs DIR
            after the K timed steps, rank 0 writes the exported columns of its
            worlds as they stand after the last timed step (what run() hands a
            caller, plus the rendered views) to DIR/<name>.npy: float32 columns
            as they are, integer columns as float64 (exact), RGBA8 as float32.
            A column over its share of 64 MiB is a fixed seeded sample of its
            rows.  Actions and world seeds are fixed, so two builds given the
            same arguments can be compared output for output.
  cpu_baseline / --impl reference
            the reference's own CPU backend (oracle/_ref, built from the
            reference sources) running the same fixture on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# workload -> (sim, worlds per GPU, sim cfg, reference-arm worlds (CPU tmp allocator is
# 32 MiB/world: include/madrona/state.hpp:362, so the CPU arm runs a bounded sample))
WORKLOADS = {
    "gridworld": dict(sim="gridworld", worlds=65536,
                      cfg={"grid_size": 8, "episode_len": 50, "init_items": 12, "seed": 0},
                      ref_worlds=1024, ref_steps=12000, taskgraphs=[0],
                      desc="pure-ECS grid sim (BASELINE configs[4] class): 2 agents + <=24 items/world, "
                           "create/destroy + compaction sort every step"),
    "cartpole": dict(sim="cartpole", worlds=65536, cfg={"max_steps": 200, "seed": 0},
                     ref_worlds=1024, ref_steps=30000, taskgraphs=[0],
                     desc="Cartpole-like fixture (BASELINE configs[0] class)"),
}
DEFAULT_WORKLOAD = "gridworld"

try:
    from bench_workloads import EXTRA_WORKLOADS, EXTRA_DEFAULT  # physics workloads
    WORKLOADS.update(EXTRA_WORKLOADS)
    DEFAULT_WORKLOAD = EXTRA_DEFAULT or DEFAULT_WORKLOAD
except ImportError:
    pass


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None

    def _loop(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                    capture_output=True, text=True, timeout=5).stdout.strip()
                parts = [p.strip() for p in out.split(",")]
                self.samples.append(float(parts[0]))
                self.max_mhz = float(parts[1])
                for nm, v in zip(names, parts[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=6)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


N_ACT = 16   # length of the action cycle both arms replay
DUMP_BYTES = 64 << 20   # all dumped columns together


def dump_outputs(ex, desc, W, cfg, render, out_dir):
    """Writes the exported columns (and rendered views) to out_dir/<name>.npy; see --dump-outputs."""
    cols = [(s.name, s.slot, s.dtype, ((ex.exportedNumRows(s.slot) if s.dynamic else W),) + s.per_world)
            for s in desc.outputs]
    if render:
        res, views = int(cfg.get("resolution", 64)), ex.exportedNumRows(14)
        cols.append(("depth", 14, "float32", (views, res, res)))
        if cfg.get("rgbd"):
            cols.append(("rgba", 13, "uint8", (views, res, res, 4)))
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // len(cols)
    for name, slot, dtype, shape in cols:
        arr = ex.tensor(slot, dtype, shape).cpu().numpy() if shape[0] else np.zeros(shape, dtype)
        arr = arr.astype(np.float64 if np.issubdtype(arr.dtype, np.integer) and arr.itemsize > 1
                         else np.float32)
        row_bytes = max(arr[:1].nbytes, 1)
        if arr.nbytes > cap:
            keep = cap // row_bytes
            arr = arr[np.sort(np.random.default_rng(0).choice(len(arr), size=keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def make_actions(desc, sim, W, steps, seed):
    rng = np.random.default_rng(seed)
    out = {}
    for s in desc.inputs:
        if s.name == "reset":
            out[s.name] = np.zeros((steps, W) + s.per_world, dtype=s.dtype)
        elif sim == "cartpole":
            out[s.name] = rng.integers(0, 2, size=(steps, W) + s.per_world).astype(s.dtype)
        elif sim == "gridworld":
            out[s.name] = rng.integers(0, 5, size=(steps, W) + s.per_world).astype(s.dtype)
        elif sim == "room":
            amount = rng.integers(0, 4, size=(steps, W, 2))
            angle = rng.integers(0, 8, size=(steps, W, 2))
            rot = rng.integers(0, 5, size=(steps, W, 2))
            out[s.name] = np.stack([amount, angle, rot], axis=-1).astype(s.dtype)
        elif sim == "arena":
            shape = (steps, W, 6)
            out[s.name] = np.stack([rng.integers(0, 4, size=shape), rng.integers(0, 8, size=shape),
                                    rng.integers(0, 5, size=shape),
                                    (rng.random(shape) < 0.1).astype(np.int64)], axis=-1).astype(s.dtype)
        else:
            out[s.name] = rng.integers(0, 4, size=(steps, W) + s.per_world).astype(s.dtype)
    return out


# what actually bounds the dominant kernel (ncu summaries under profiles/); the JSON
# contract only knows "hbm" / "tensor", so the HBM fraction is always reported
_LATENCY = ("per-world / per-candidate kernel: one wave whose duration is the slowest world's dependent chain; "
            "instruction-issue / latency bound (ncu round 2, profiles/r2c_ncu_summary.txt: 19-43 % issue "
            "utilisation, 18-35 % achieved occupancy), as SURVEY 8d anticipated; the HBM fraction is reported "
            "for completeness")
ROOFLINE_NOTES = {
    "phys_narrowphase": _LATENCY, "phys_solve_positions": _LATENCY, "phys_solve_velocities": _LATENCY,
    "phys_find_candidates": _LATENCY,
    "raycast": "instruction bound (ncu: 71 % issue utilisation, 30 active threads per instruction); algorithmic "
               "bytes = the 8 B written per pixel",
    "sort_archetype": "whole sort (histogram + P onesweep passes + column-major gather + copy-back); a random "
                      "row permutation makes the gather and the entity re-pointing latency bound (ncu: 58 % "
                      "long-scoreboard stalls), each onesweep pass is bound by its per-tile serial phases "
                      "(DESIGN.md 3.1)",
    "compact_archetype": "whole compaction sort (histogram + P onesweep passes + column-major gather + copy-back)",
}


def run_reference_arm(args, wl, reps=3):
    """The reference's own CPU implementation of the path on the host cores,
    replaying the SAME seeded action tensor as the GPU arm (its first
    `ref_worlds` worlds, the same 16-step cycle)."""
    from oracle import runner
    from sims import SIMS

    desc = SIMS[wl["sim"]]
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    W = wl["ref_worlds"]
    if not W:
        return None   # GPU-only microbenchmark: no CPU-backend counterpart
    # a bounded sample of the workload that is long enough for the CPU backend's
    # cold start (thread pool, first BVH build) to be amortised -- with only K+W
    # simulation steps the reference would be timed mostly cold
    steps = getattr(args, "ref_steps", None) or max(args.steps + args.warmup, wl.get("ref_steps", 2000))
    if not runner.available(desc.name):
        return None
    cycle = make_actions(desc, wl["sim"], wl["worlds"], N_ACT, seed=1000)
    inputs = None
    if desc.inputs:
        idx = np.arange(steps) % N_ACT
        inputs = {k: np.ascontiguousarray(v[idx][:, :W]) for k, v in cycle.items()}
    runs, walls = [], []
    for _ in range(reps):
        t0 = time.time()
        _, timing = runner.run_reference(desc, W, steps, inputs, wl["cfg"], workers=cores, want_outputs=False)
        walls.append(time.time() - t0)
        runs.append(timing)
    order = sorted(range(reps), key=lambda i: runs[i]["steps_per_sec"])
    med = runs[order[reps // 2]]
    vals = [r["steps_per_sec"] for r in runs]
    return {"value": med["steps_per_sec"], "unit": "env-steps/s", "cores": cores, "kind": "reference",
            "sample": f"{desc.name}: {W} worlds x {steps} steps (RAM-bounded: the CPU backend's tmp allocator is "
                      f"32 MiB/world, include/madrona/state.hpp:362), reference TaskGraphExecutor "
                      f"numWorkers={cores} (oracle/_ref, g++ -O2 -march=x86-64-v3), same seeded random actions as "
                      f"the GPU arm (first {W} worlds, {N_ACT}-step cycle); median of {reps} runs, "
                      f"min/max {min(vals):.0f}/{max(vals):.0f} env-steps/s, "
                      f"{med['seconds']:.2f}s in run() / {walls[order[reps // 2]]:.1f}s wall",
            "runs": vals,
            "ms_per_step": med["seconds"] / steps * 1e3, "worlds": W}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--worlds", type=int, default=0, help="worlds per GPU (default: workload's)")
    ap.add_argument("--no-l2-flush", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: NVLink peer-store gather kernel (default) or one packed NCCL all_gather per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (rank 0's worlds)")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    if args.worlds:
        wl["worlds"] = args.worlds

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))

    metric = "aggregate env-steps/sec"
    config = {"workload": f"{args.workload}: {wl['desc']}", "worlds_per_gpu": wl["worlds"],
              "sim_cfg": wl["cfg"], "parallelism": f"world-shard x{world_size}"}

    if args.impl == "reference":
        if rank != 0:
            return
        res = run_reference_arm(args, wl)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built on this box"}))
            return
        line = {"impl": "reference", "metric": metric, "value": res["value"], "unit": "env-steps/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+i32", "data": "synthetic",
                "config": dict(config, worlds_per_gpu=res["worlds"]),
                "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "runs")},
                "e2e": {"value": res["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    from sims import SIMS, make_executor

    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_size > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    desc = SIMS[wl["sim"]]
    W = wl["worlds"]
    from madrona_b200 import sharding
    first_world, _ = sharding.shard_range(W * world_size, world_size, rank)
    cfg = dict(wl["cfg"])
    # world seeds depend on the GLOBAL world index: rank r simulates worlds [r*W, (r+1)*W)
    cfg["seed"] = sharding.world_seed(int(cfg.get("seed", 0)), first_world, 0)
    ex = make_executor(wl["sim"], W, gpu_id=local_rank, **cfg)
    graph = ex.buildLaunchGraph(wl["taskgraphs"])
    launches_per_step = graph.num_kernels
    render_graph = ex.buildRenderGraph() if wl.get("render") else None
    if render_graph is not None:
        launches_per_step += render_graph.num_kernels

    in_t = {s.name: ex.tensor(s.slot, s.dtype, (W,) + s.per_world) for s in desc.inputs}
    fixed_out = [s for s in desc.outputs if not s.dynamic and s.name in ("reward", "done")]
    out_t = {s.name: ex.tensor(s.slot, s.dtype, (W,) + s.per_world) for s in fixed_out}

    n_act = N_ACT
    host_actions = make_actions(desc, wl["sim"], W, n_act, seed=1000 + rank)
    dev_actions = {k: torch.from_numpy(v).to(dev) for k, v in host_actions.items()}
    pinned_actions = {k: torch.from_numpy(v).pin_memory() for k, v in host_actions.items()}
    pinned_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out_t.items()}

    stream = torch.cuda.current_stream()
    flush = None if args.no_l2_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---- N > 1: the gather of the exported reward / done columns
    gather_kind = None
    pg = None
    nccl = None
    if world_size > 1 and out_t:
        if args.gather == "p2p":
            try:
                pg = ex.peerGather([s.slot for s in fixed_out], [(W,) + s.per_world for s in fixed_out],
                                   [s.dtype for s in fixed_out], world_size, rank)
                sharding.connect_peer_gather(pg)
                gather_kind = "p2p-push: one NVLink peer-store kernel per rank per step into every peer's " \
                              "symmetric buffer, consumed one step later (peer_gather.cu)"
            except Exception as e:      # e.g. cudaIpc refused by the container
                pg = None
                gather_kind = f"nccl (p2p unavailable: {e})"
        ok = torch.tensor([1 if pg is not None or args.gather == "nccl" else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0 or args.gather == "nccl":
            if pg is not None:
                pg.close()
                pg = None
            # ONE packed all_gather per step on a side stream, double buffered
            pack_elems = sum(t.numel() for t in out_t.values())   # all 4-byte columns
            nccl = dict(side=torch.cuda.Stream(device=dev),
                        pack=[torch.empty(pack_elems, dtype=torch.int32, device=dev) for _ in range(2)],
                        out=[torch.empty(world_size * pack_elems, dtype=torch.int32, device=dev) for _ in range(2)],
                        done_ev=[torch.cuda.Event() for _ in range(2)],
                        packed_ev=[torch.cuda.Event() for _ in range(2)])
            gather_kind = gather_kind or "nccl: one packed all_gather_into_tensor per step on a side stream, " \
                                         "double buffered"
            # warm NCCL (channel setup, first-use allocations) outside the --warmup budget
            for _ in range(64):
                dist.all_gather_into_tensor(nccl["out"][0], nccl["pack"][0])
            torch.cuda.synchronize()
    p2p = None
    if pg is not None:
        p2p = dict(side=torch.cuda.Stream(device=dev), done_ev=[torch.cuda.Event() for _ in range(2)],
                   pushed_ev=[torch.cuda.Event() for _ in range(2)])
    step_counter = [0]

    def gather_step():
        k = step_counter[0]
        step_counter[0] += 1
        if pg is not None:
            # the gather runs on a side stream: the compute stream only waits until its
            # columns have been read (push done), not for the peers
            par = k & 1
            p2p["done_ev"][par].record(stream)
            side = p2p["side"]
            side.wait_event(p2p["done_ev"][par])
            pg.push(side)
            p2p["pushed_ev"][par].record(side)
            if k >= 1:
                pg.wait(side)       # step k-1 of every rank has landed here
                pg.release(side)    # (a learner would read pg.tensor((k-1) & 1, i) in between)
            stream.wait_event(p2p["pushed_ev"][par])
        elif nccl is not None:
            par = k & 1
            nccl["done_ev"][par].record(stream)
            with torch.cuda.stream(nccl["side"]):
                nccl["side"].wait_event(nccl["done_ev"][par])
                torch.cat([t.reshape(-1).view(torch.int32) for t in out_t.values()], out=nccl["pack"][par])
                nccl["packed_ev"][par].record(nccl["side"])
                dist.all_gather_into_tensor(nccl["out"][par], nccl["pack"][par])
            # the next step graph may overwrite the columns once they are packed
            stream.wait_event(nccl["packed_ev"][par])

    def gather_drain():
        if pg is not None and step_counter[0] >= 1:
            pg.wait(p2p["side"])
            pg.release(p2p["side"])
            stream.wait_stream(p2p["side"])
        if nccl is not None:
            stream.wait_stream(nccl["side"])

    def one_step(i, host_io=False):
        if host_io:
            for k, t in in_t.items():
                t.copy_(pinned_actions[k][i % n_act], non_blocking=True)
        else:
            for k, t in in_t.items():
                t.copy_(dev_actions[k][i % n_act], non_blocking=True)
        ex.runAsync(graph, stream)
        if render_graph is not None:
            ex.runAsync(render_graph, stream)
        if world_size > 1:
            gather_step()
        if host_io:
            for k, t in out_t.items():
                pinned_out[k].copy_(t, non_blocking=True)

    def timed(host_io):
        for i in range(args.warmup):
            one_step(i, host_io)
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        for i in range(args.steps):
            if flush is not None:
                flush.fill_(i & 0xff)
            starts[i].record(stream)
            one_step(i, host_io)
            ends[i].record(stream)
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()
        per_step = np.array([s.elapsed_time(e) for s, e in zip(starts, ends)])
        total_ms = float(per_step.sum())
        t = torch.tensor([total_ms, float(per_step.min()), float(np.median(per_step)), float(per_step.max())],
                         dtype=torch.float64, device=dev)
        if world_size > 1:
            allr = [torch.empty_like(t) for _ in range(world_size)]
            dist.all_gather(allr, t)
            stats = [[round(float(v), 4) for v in r.tolist()] for r in allr]
            total_ms = max(r[0] for r in stats)
        else:
            stats = [[round(float(v), 4) for v in t.tolist()]]
        return total_ms, stats

    def run_loop_wall():
        """Plain wall clock of K back-to-back run() calls (launch + stream sync each), no flush."""
        for i in range(3):
            ex.run(graph)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(args.steps):
            ex.run(graph)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    total_ms, rank_stats = timed(host_io=False)
    if args.dump_outputs and rank == 0:
        torch.cuda.synchronize()
        dump_outputs(ex, desc, W, cfg, render_graph is not None, args.dump_outputs)
    e2e_ms, e2e_rank_stats = timed(host_io=True)
    if world_size > 1:
        gather_drain()
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    wall_ms = run_loop_wall() if world_size == 1 else None

    h2d = sum(int(np.prod(v.shape[1:])) * v.dtype.itemsize for v in host_actions.values())
    d2h = sum(t.numel() * t.element_size() for t in out_t.values())

    roofline = None
    cpu_base = None
    if rank == 0:
        peak, peak_kind = load_peaks()
        prof = ex.profileNodes(wl["taskgraphs"], reps=20)
        prof = [p for p in prof if p["bytes"] > 0 and p["ms"] > 0]
        if render_graph is not None:
            # the ray caster is its own launch graph: time it with events on the same stream
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            reps = 10
            ex.runAsync(render_graph, stream)
            evs[0].record(stream)
            for _ in range(reps):
                ex.runAsync(render_graph, stream)
            evs[1].record(stream)
            torch.cuda.synchronize()
            res = int(cfg.get("resolution", 64))
            views = ex.exportedNumRows(14)
            per_px = 8 if cfg.get("rgbd") else 4
            prof.append({"kind": "raycast", "node": -1, "ms": evs[0].elapsed_time(evs[1]) / reps,
                         "rows": float(views), "bytes": float(views * res * res * per_px)})
        if prof:
            # dominant kernel = the node kind with the largest share of the step
            kinds = {}
            for p in prof:
                k = kinds.setdefault(p["kind"], {"ms": 0.0, "bytes": 0.0, "rows": 0.0, "launches": 0})
                k["ms"] += p["ms"]
                k["bytes"] += p["bytes"]
                k["rows"] += p["rows"]
                k["launches"] += 1
            top_kind = max(kinds, key=lambda k: kinds[k]["ms"])
            top = kinds[top_kind]
            ms_per_launch = top["ms"] / top["launches"]
            bytes_per_launch = top["bytes"] / top["launches"]
            gbs = bytes_per_launch / (ms_per_launch * 1e-3) / 1e9
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tpath):
                # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed
                # `ncu --set full` capture of this workload (profiles/*_ncu_summary.csv)
                traffic = json.load(open(tpath)).get(args.workload, {}).get(top_kind)
            step_ms = sum(k["ms"] for k in kinds.values())
            roofline = {"bound": "hbm", "kernel": top_kind, "launches_per_step": top["launches"],
                        "share_of_step": top["ms"] / step_ms,
                        "achieved": gbs, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                        "frac": gbs / peak, "traffic": traffic,
                        "algorithmic_bytes_per_launch": bytes_per_launch, "ms_per_launch": ms_per_launch,
                        "units_per_launch": top["rows"] / top["launches"],
                        "note": ROOFLINE_NOTES.get(top_kind, ""),
                        "all_kinds": [{"kind": k, "launches": v["launches"], "ms_total": round(v["ms"], 5),
                                       "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)}
                                      for k, v in kinds.items()]}
        if world_size == 1 and not args.no_cpu_baseline:
            # bounded sample: ~10-20 s of CPU work on the box's host cores
            small = argparse.Namespace(steps=0, warmup=0, ref_steps=wl.get("ref_steps", 2000))
            res = run_reference_arm(small, wl)
            if res:
                cpu_base = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "runs")}

    if pg is not None:
        pg.close()
    ex.close()
    if rank == 0:
        total_worlds = W * world_size
        line = {
            "metric": metric,
            "value": total_worlds * args.steps / (total_ms * 1e-3),
            "unit": "env-steps/s",
            "n_gpus": world_size,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32+i32",
            "data": "synthetic",
            "config": dict(config, l2="flushed between steps (256 MiB write)" if flush is not None
                           else "not flushed"),
            "timing": "sum of per-step CUDA-event intervals on the launching stream (L2 flush between steps "
                      "excluded), max over ranks",
            "run_loop": None if wall_ms is None else {
                "value": total_worlds * args.steps / (wall_ms * 1e-3), "unit": "env-steps/s",
                "ms_per_step": wall_ms / args.steps,
                "what": "wall clock of K back-to-back run() calls (graph launch + stream sync), no L2 flush"},
            "gather": None if world_size == 1 else {
                "kind": gather_kind, "bytes_per_rank_per_step": d2h,
                "per_rank_ms [total, step min, median, max]": rank_stats,
                "per_rank_ms_e2e": e2e_rank_stats},
            "clocks": clocks,
            "e2e": {"value": total_worlds * args.steps / (e2e_ms * 1e-3), "unit": "env-steps/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches_per_step) * args.steps,
            "roofline": roofline,
            "cpu_baseline": cpu_base,
        }
        print(json.dumps(line))
    if world_size > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
