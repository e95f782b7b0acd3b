#!/usr/bin/env bash
# Round 6, second call: the other workloads once per build (this tree's library and the parent commit's), both builds'
# --dump-outputs compared on each of them, then the whole GPU suite.
# usage: bash scripts/gpu_r6_others.sh <parent build> <output directory>
set -u
PARENT=$1; OUT=$2
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1; cat "$OUT/gpu.csv"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || exit 1
BENCH="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline"
for w in cfg4_fill_sphere10M_4k_16spp cfg5_hair1M_4k cfg1_robot_720p cfg2_robot_textured_720p_4spp cfg3_robot_reflect16_1080p; do
    $BENCH --workload "$w" > "$OUT/new_$w.json" 2> "$OUT/new_$w.log"
    $BENCH --workload "$w" --lib "$PARENT" > "$OUT/old_$w.json" 2> "$OUT/old_$w.log"
    $BENCH --workload "$w" --steps 3 --no-ref-work --dump-outputs "$OUT/dn" > /dev/null 2>> "$OUT/dump.log"
    $BENCH --workload "$w" --steps 3 --no-ref-work --dump-outputs "$OUT/do" --lib "$PARENT" > /dev/null 2>> "$OUT/dump.log"
    python - "$OUT" "$w" <<'PY'
import sys, numpy as np
out, w = sys.argv[1], sys.argv[2]
for f in ("frame.npy", "ray_counts.npy", "frame_pixels.npy"):
    a, b = np.load(f"{out}/dn/{f}"), np.load(f"{out}/do/{f}")
    print(w, f, "identical" if a.shape == b.shape and np.array_equal(a, b) else "DIFFERENT")
PY
    rm -rf "$OUT/dn" "$OUT/do"
done
python - "$OUT" <<'PY'
import glob, json, os, sys
out = sys.argv[1]
for f in sorted(glob.glob(f"{out}/*.json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:
        print(os.path.basename(f), "no result", e); continue
    st = d["roofline"]["stage_ms_per_step"]
    print(f"{os.path.basename(f):48s} {d['ms_per_step']:8.3f} ms  primary {st['k_primary']:.3f} shade {st['k_shade']:.3f} "
          f"build {d['bvh']['build_ms']:.1f} ms  clock {d['clocks'].get('sm_mhz')}")
PY
timeout 1800 python -m pytest -q -m gpu > "$OUT/pytest_gpu_all.log" 2>&1; echo "gpu suite rc $?"
tail -5 "$OUT/pytest_gpu_all.log"
