#!/usr/bin/env bash
# Round 5 (screen coverage of the primary packets) on one GPU: smoke, the GPU tests of the coverage, the A/B of this tree's
# library against the parent commit's build (scripts/gpu_ab_bench.sh), the cost of a camera move against the parent, the
# coverage rebuild and upload on their own (RTB200_TRACE), then the whole GPU suite.
# usage: bash scripts/gpu_r5_screen_coverage.sh <parent build of librtb200.so> <output directory>
set -u
OTHER=$1; OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc $?"
python -m pytest -q tests/test_screen_coverage.py > "$OUT/pytest_coverage.log" 2>&1; echo "coverage tests rc $?"
tail -3 "$OUT/pytest_coverage.log"
bash scripts/gpu_ab_bench.sh "$OTHER" "$OUT/ab" 3 > "$OUT/ab.txt" 2>&1; echo "ab rc $?"
cat "$OUT/ab.txt"
python scripts/gpu_camera_move.py > "$OUT/camera_move_new.json" 2> "$OUT/camera_move_new.log"; echo "camera move rc $?"
python scripts/gpu_camera_move.py --lib "$OTHER" > "$OUT/camera_move_old.json" 2> "$OUT/camera_move_old.log"; echo "camera move (parent) rc $?"
cat "$OUT/camera_move_new.json" "$OUT/camera_move_old.json"
RTB200_TRACE=1 python scripts/gpu_camera_move.py --moves 2 2>&1 | grep -E "screen coverage|wide tree" > "$OUT/coverage_trace.txt"
head -6 "$OUT/coverage_trace.txt"
timeout 1500 python -m pytest -q -m gpu > "$OUT/pytest_gpu_all.log" 2>&1; echo "gpu suite rc $?"
tail -5 "$OUT/pytest_gpu_all.log"
