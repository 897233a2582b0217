#!/bin/bash
# (Record only: MADRONA_B200_SORT_FUSE_COPYBACK and the MADRONA_B200_*_BLOCKS_PER_SM switches used below no longer exist.)
# Round-2 batch B (one gpurun call): parity of the new kernels, bench lines, one-box A/Bs of
# every switch added since batch A, then ncu captures (last: a killed ncu can wedge a GPU).
# Variant libraries used below were built beforehand (git-ignored) with
#   scripts/build_variants.sh bodyold "-DMB2_BODY_MINB=1" look1 "-DMB2_SORT_LOOK_WINDOW=1" sort12 "-DMB2_SORT_ITEMS=12" \
#       sort16 "-DMB2_SORT_ITEMS=16" rc2 "-DMB2_RAYCAST_MINB=2"
# at commit 0b970f5 (the defaults of that commit: fused copy-back ON, 32-register row kernels, traceRay seed ON).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
T0=$(date +%s)
stamp() { echo "== $1 @ $(( $(date +%s) - T0 ))s"; }
L=madrona_b200
timeout 900 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider 2>&1 | tail -60 > gpurun_out/r2b_pytest_gpu.txt
tail -15 gpurun_out/r2b_pytest_gpu.txt
stamp pytest
if ! grep -q " passed" gpurun_out/r2b_pytest_gpu.txt || grep -q "failed" gpurun_out/r2b_pytest_gpu.txt; then
  echo "-- failures: re-run the physics / sort fixtures with each new switch off"
  MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_SEED=0 timeout 400 python -m pytest tests/test_room.py tests/test_arena.py -m gpu -q --tb=line -p no:cacheprovider 2>&1 | tail -8
  MADRONA_B200_SORT_FUSE_COPYBACK=0 timeout 400 python -m pytest tests/test_sort_custom_key.py tests/test_gridworld.py tests/test_room.py -m gpu -q --tb=line -p no:cacheprovider 2>&1 | tail -8
  stamp pytest_attribution
fi
run() {   # label workload [ENV=VAL ...]
  local label=$1 wl=$2; shift 2
  env "$@" timeout 200 python bench.py --workload $wl --steps 100 --warmup 10 --no-cpu-baseline 2>gpurun_out/err_$label.txt \
    | tail -1 > gpurun_out/r2b_bench_$label.json
  python - "$label" <<'PY'
import json, sys
try:
    d = json.loads(open(f"gpurun_out/r2b_bench_{sys.argv[1]}.json").read())
    r = d.get("roofline") or {}
    print("%-28s ms/step %.4f  e2e %.4f  top %s frac %.3f" % (sys.argv[1], d["ms_per_step"], d["e2e"]["ms_per_step"],
          r.get("kernel"), r.get("frac") or 0))
except Exception as e:
    print(sys.argv[1], "FAILED", e)
PY
}
for wl in room arena sortcheck gridworld room_render; do run $wl $wl X=1; done
stamp benches
run room_noseed room MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_SEED=0
run room_body4 room MADRONA_B200_BODY_BLOCKS_PER_SM=4
run room_bodyold room MADRONA_B200_LIB=$L/libmadrona_b200_bodyold.so MADRONA_B200_BODY_BLOCKS_PER_SM=4
run arena_noseed arena MADRONA_B200_JIT_DEFINES=-DMB2_TRACE_SEED=0
run room_2 room X=1
stamp ab_room
run sort_nofuse sortcheck MADRONA_B200_SORT_FUSE_COPYBACK=0
run sort_move4 sortcheck MADRONA_B200_REARRANGE_BLOCKS_PER_SM=4
run sort_look1 sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_look1.so
run sort_items12 sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_sort12.so
run sort_items16 sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_sort16.so
run sort_items16_3 sortcheck MADRONA_B200_LIB=$L/libmadrona_b200_sort16.so MADRONA_B200_SWEEP_BLOCKS_PER_SM=3
run sort_2 sortcheck X=1
run render_minb2 room_render MADRONA_B200_LIB=$L/libmadrona_b200_rc2.so
run render_2 room_render X=1
stamp ab_sort_render
timeout 200 ncu --metrics gpu__time_duration.sum --clock-control none --launch-skip 700 -c 140 --csv \
  --log-file gpurun_out/r2b_launches_room.csv python bench.py --workload room --steps 12 --warmup 4 --no-cpu-baseline \
  > gpurun_out/ncu_launch_room.log 2>&1
stamp launch_list
timeout 200 ncu --set full --import-source on --clock-control none -k regex:"sort" --launch-skip 14 --launch-count 7 -f \
  -o gpurun_out/r2b_sort python bench.py --workload sortcheck --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_sort.log 2>&1
stamp ncu_sort
timeout 200 ncu --set full --import-source on --clock-control none -k regex:"nodeKern" --launch-skip 14 --launch-count 7 -f \
  -o gpurun_out/r2b_nodes python bench.py --workload room --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_nodes.log 2>&1
stamp ncu_nodes
timeout 240 ncu --set full --import-source on --clock-control none -k regex:"phys" --launch-skip 84 --launch-count 30 -f \
  -o gpurun_out/r2b_phys python bench.py --workload room --steps 3 --warmup 2 --no-cpu-baseline > gpurun_out/ncu_phys.log 2>&1
stamp ncu_phys
timeout 240 ncu --set full --import-source on --clock-control none -k regex:"renderRaycast" --launch-skip 2 --launch-count 2 -f \
  -o gpurun_out/r2b_render python bench.py --workload room_render --worlds 1024 --steps 2 --warmup 1 --no-cpu-baseline > gpurun_out/ncu_render.log 2>&1
stamp ncu_render
ls -la gpurun_out/*.ncu-rep
du -sh gpurun_out
