#!/usr/bin/env bash
# A/B of this tree's library against another build of it on one GPU: bench.py alternated between the two, RUNS times each
# on the headline workload (OUT/{new,old}_<i>.json), the outputs of both dumped (must be identical), the packet round
# histograms of the instrumented kernels (RTB200_TRACE, OUT/trace_*.log), then the other workloads once per build.
# usage: bash scripts/gpu_ab_bench.sh <other build of librtb200.so> <output directory> [RUNS] [workload ...]
set -u
OTHER=$1; OUT=$2; RUNS=${3:-3}; shift 2; shift || true
OTHERS=${*:-"cfg4_fill_sphere10M_4k_16spp cfg5_hair1M_4k cfg1_robot_720p cfg2_robot_textured_720p_4spp cfg3_robot_reflect16_1080p"}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1
python -c "import __graft_entry__ as g; g.build()" || exit 1
BENCH="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline"
for i in $(seq "$RUNS"); do
    $BENCH > "$OUT/new_$i.json" 2> "$OUT/new_$i.log"
    $BENCH --lib "$OTHER" > "$OUT/old_$i.json" 2> "$OUT/old_$i.log"
done
$BENCH --steps 3 --no-ref-work --dump-outputs "$OUT/dump_new" > /dev/null 2> "$OUT/dump_new.log"
$BENCH --steps 3 --no-ref-work --dump-outputs "$OUT/dump_old" --lib "$OTHER" > /dev/null 2> "$OUT/dump_old.log"
python - "$OUT" <<'EOF'
import sys, numpy as np
out = sys.argv[1]
for f in ("frame.npy", "ray_counts.npy", "frame_pixels.npy"):
    a, b = np.load(f"{out}/dump_new/{f}"), np.load(f"{out}/dump_old/{f}")
    print(f, "identical" if a.shape == b.shape and np.array_equal(a, b) else "DIFFERENT")
EOF
rm -rf "$OUT/dump_new" "$OUT/dump_old"                                         # ~50 MB each
RTB200_TRACE=1 $BENCH --steps 1 --no-ref-work > /dev/null 2> "$OUT/trace_new.log"
RTB200_TRACE=1 $BENCH --steps 1 --no-ref-work --lib "$OTHER" > /dev/null 2> "$OUT/trace_old.log"
grep -E "wide tree|octree:|packets .* histogram|split (shadow|primary)" "$OUT/trace_new.log" "$OUT/trace_old.log"
for w in $OTHERS; do
    $BENCH --workload "$w" > "$OUT/new_$w.json" 2> "$OUT/new_$w.log"
    $BENCH --workload "$w" --lib "$OTHER" > "$OUT/old_$w.json" 2> "$OUT/old_$w.log"
done
python - "$OUT" <<'EOF'
import glob, json, os, sys
out = sys.argv[1]
for f in sorted(glob.glob(f"{out}/*.json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:
        print(os.path.basename(f), "no result", e); continue
    st = d["roofline"]["stage_ms_per_step"]
    print(f"{os.path.basename(f):50s} {d['ms_per_step']:8.3f} ms  primary {st['k_primary']:.3f} shade {st['k_shade']:.3f} "
          f"build {d['bvh']['build_ms']:.1f} ms  fetched p/s {d['work']['primary_fetched_bytes']}/{d['work']['shadow_fetched_bytes']}  "
          f"clock {d['clocks'].get('sm_mhz')}")
EOF
