#!/bin/bash
# (Record only: -DMB2_TRACE_MASK=0, MADRONA_B200_SORT_FUSE_COPYBACK and MADRONA_B200_REARRANGE_BLOCKS_PER_SM used below no longer exist.)
# Round-2 batch C (one gpurun call): parity, one-box A/Bs of the last switches (traceRay candidate
# mask, ballot digit matching, rearrange residency), then the bench lines and ncu captures of the
# configuration the A/Bs select (recorded in gpurun_out/r2c_selected.env), ncu last.
# The ballot variant was built beforehand (git-ignored) with
#   scripts/build_variants.sh ballot "-DMB2_SORT_MATCH_BALLOT=1"      (commit c1ae823; that code path was removed afterwards)
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
T0=$(date +%s)
stamp() { echo "== $1 @ $(( $(date +%s) - T0 ))s"; }
L=madrona_b200
timeout 900 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider 2>&1 | tail -60 > gpurun_out/r2c_pytest_gpu.txt
tail -12 gpurun_out/r2c_pytest_gpu.txt
stamp pytest
MADRONA_B200_LIB=$L/libmadrona_b200_ballot.so timeout 400 python -m pytest tests/test_sort_custom_key.py tests/test_gridworld.py \
  tests/test_full_size.py tests/test_room.py -m gpu -q --tb=line -p no:cacheprovider 2>&1 | tail -4 | tee gpurun_out/r2c_pytest_ballot.txt
MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_MASK=0 timeout 300 python -m pytest tests/test_room.py tests/test_arena.py -m gpu -q --tb=line \
  -p no:cacheprovider 2>&1 | tail -3 | tee gpurun_out/r2c_pytest_walk.txt
stamp pytest_variants

run() {   # label workload [ENV=VAL ...]
  local label=$1 wl=$2; shift 2
  env "$@" timeout 200 python bench.py --workload $wl --steps 100 --warmup 10 --no-cpu-baseline 2>gpurun_out/err_$label.txt \
    | tail -1 > gpurun_out/r2c_bench_$label.json
  python - "$label" <<'PY'
import json, sys
try:
    d = json.loads(open(f"gpurun_out/r2c_bench_{sys.argv[1]}.json").read())
    r = d.get("roofline") or {}
    print("%-28s ms/step %.4f  e2e %.4f  top %s frac %.3f" % (sys.argv[1], d["ms_per_step"], d["e2e"]["ms_per_step"],
          r.get("kernel"), r.get("frac") or 0))
except Exception as e:
    print(sys.argv[1], "FAILED", e)
PY
}
ms() { python -c "import json,sys; print(json.loads(open('gpurun_out/r2c_bench_%s.json' % sys.argv[1]).read())['ms_per_step'])" $1 2>/dev/null || echo 1e9; }

run room_mask room X=1
run room_walk room MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_MASK=0
run arena_mask arena X=1
run arena_walk arena MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_MASK=0
run room_mask2 room X=1
run room_walk2 room MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_MASK=0
stamp ab_trace
run sort_match sortcheck X=1
run sort_ballot sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_ballot.so
run sort_move5 sortcheck MADRONA_B200_REARRANGE_BLOCKS_PER_SM=5
run sort_move8 sortcheck MADRONA_B200_REARRANGE_BLOCKS_PER_SM=8
run sort_fuse sortcheck MADRONA_B200_SORT_FUSE_COPYBACK=1
run sort_match2 sortcheck X=1
run sort_ballot2 sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_ballot.so
run grid_match gridworld X=1
run grid_ballot gridworld MADRONA_B200_LIB=$L/libmadrona_b200_ballot.so
stamp ab_sort

# ---- select (the faster of each pair, both repetitions summed)
SEL=""
python - > gpurun_out/r2c_selected.env <<'PY'
import json
def ms(l):
    try: return json.loads(open(f"gpurun_out/r2c_bench_{l}.json").read())["ms_per_step"]
    except Exception: return 1e9
env = []
if ms("room_walk") + ms("room_walk2") + 0.2 * ms("arena_walk") < ms("room_mask") + ms("room_mask2") + 0.2 * ms("arena_mask"):
    env.append("MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_MASK=0")
if ms("sort_ballot") + ms("sort_ballot2") < ms("sort_match") + ms("sort_match2"):
    env.append("MADRONA_B200_LIB=madrona_b200/libmadrona_b200_ballot.so")
best = min(("6", ms("sort_match") + ms("sort_match2")), ("5", 2 * ms("sort_move5")), ("8", 2 * ms("sort_move8")), key=lambda t: t[1])
if best[0] != "6":
    env.append("MADRONA_B200_REARRANGE_BLOCKS_PER_SM=" + best[0])
print(" ".join(env) if env else "X=1")
PY
SEL=$(cat gpurun_out/r2c_selected.env)
echo "selected: $SEL"

# ---- final lines with the selected configuration
env $SEL timeout 300 python bench.py 2>gpurun_out/err_final_room.txt | tail -1 > gpurun_out/r2c_final_room.json
for wl in arena sortcheck gridworld room_render; do
  env $SEL timeout 200 python bench.py --workload $wl --steps 100 --warmup 10 --no-cpu-baseline 2>gpurun_out/err_final_$wl.txt \
    | tail -1 > gpurun_out/r2c_final_$wl.json
done
timeout 200 python bench.py --impl reference --steps 20 --warmup 5 2>gpurun_out/err_ref.txt | tail -1 > gpurun_out/r2c_reference_room.json
python - <<'PY'
import json
for wl in ("room", "arena", "sortcheck", "gridworld", "room_render"):
    try:
        d = json.loads(open(f"gpurun_out/r2c_final_{wl}.json").read())
        r = d.get("roofline") or {}
        print("FINAL %-12s ms/step %.4f value %.4g e2e %.4g top %s frac %.3f cpu %s" % (wl, d["ms_per_step"], d["value"],
              d["e2e"]["value"], r.get("kernel"), r.get("frac") or 0, (d.get("cpu_baseline") or {}).get("value")))
    except Exception as e:
        print("FINAL", wl, "FAILED", e)
try:
    print("REFERENCE ARM", json.loads(open("gpurun_out/r2c_reference_room.json").read())["value"])
except Exception as e:
    print("REFERENCE ARM FAILED", e)
PY
stamp finals

# ---- ncu (last: a killed ncu can wedge a GPU)
env $SEL timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none --launch-skip 700 -c 140 --csv \
  --log-file gpurun_out/r2c_launches_room.csv python bench.py --workload room --steps 12 --warmup 4 --no-cpu-baseline \
  > gpurun_out/ncu_launch_room.log 2>&1
env $SEL timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none --launch-skip 700 -c 140 --csv \
  --log-file gpurun_out/r2c_launches_arena.csv python bench.py --workload arena --steps 12 --warmup 4 --no-cpu-baseline \
  > gpurun_out/ncu_launch_arena.log 2>&1
stamp launch_lists
env $SEL timeout 200 ncu --set full --import-source on --clock-control none -k regex:"sort" --launch-skip 14 --launch-count 7 -f \
  -o gpurun_out/r2c_sort python bench.py --workload sortcheck --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_sort.log 2>&1
stamp ncu_sort
env $SEL timeout 200 ncu --set full --import-source on --clock-control none -k regex:"nodeKern" --launch-skip 14 --launch-count 7 -f \
  -o gpurun_out/r2c_nodes python bench.py --workload room --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_nodes.log 2>&1
stamp ncu_nodes
env $SEL timeout 240 ncu --set full --clock-control none -k regex:"phys" --launch-skip 84 --launch-count 30 -f \
  -o gpurun_out/r2c_phys python bench.py --workload room --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_phys.log 2>&1
stamp ncu_phys
env $SEL timeout 200 ncu --set full --import-source on --clock-control none -k regex:"renderRaycast" --launch-skip 2 --launch-count 2 -f \
  -o gpurun_out/r2c_render python bench.py --workload room_render --worlds 1024 --steps 2 --warmup 1 --no-cpu-baseline > gpurun_out/ncu_render.log 2>&1
stamp ncu_render
ls -la gpurun_out/r2c_*.ncu-rep
du -sh gpurun_out
