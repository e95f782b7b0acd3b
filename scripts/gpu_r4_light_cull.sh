#!/usr/bin/env bash
# Round 4 (light cull of the shadow packets) on one GPU: smoke, the GPU tests of the masks and of the wide tree, the A/B of
# this tree's library against the parent commit's build (scripts/gpu_ab_bench.sh), the cost of a light move, the mask pass
# on its own (RTB200_TRACE), then the whole GPU suite.
# usage: bash scripts/gpu_r4_light_cull.sh <parent build of librtb200.so> <output directory>
set -u
OTHER=$1; OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc $?"
python -m pytest -q -m gpu tests/test_light_cull.py tests/test_wide_tree.py > "$OUT/pytest_cull_wide.log" 2>&1; echo "cull/wide tests rc $?"
tail -3 "$OUT/pytest_cull_wide.log"
bash scripts/gpu_ab_bench.sh "$OTHER" "$OUT/ab" 3 > "$OUT/ab.txt" 2>&1; echo "ab rc $?"
cat "$OUT/ab.txt"
python scripts/gpu_light_move.py > "$OUT/light_move.json" 2> "$OUT/light_move.log"; echo "light move rc $?"
cat "$OUT/light_move.json"
RTB200_TRACE=1 python scripts/gpu_light_move.py --moves 2 2>&1 | grep -E "light_mask|wide tree" > "$OUT/light_mask_trace.txt"
head -5 "$OUT/light_mask_trace.txt"
timeout 1500 python -m pytest -q -m gpu > "$OUT/pytest_gpu_all.log" 2>&1; echo "gpu suite rc $?"
tail -5 "$OUT/pytest_gpu_all.log"
