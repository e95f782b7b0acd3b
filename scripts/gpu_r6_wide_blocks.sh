#!/usr/bin/env bash
# Round 6 (blocks of up to 16 records in the wide tree) on one GPU: smoke, the GPU tests of the wide tree, the light cull and
# the screen coverage, the headline frame alternated three times between this tree's library (16), builds of it with
# kWideBlock 12 and 8, and the parent commit's library; both dumps compared; the packet round histograms and block levels
# (RTB200_TRACE) of each build; the stack bound of the nested test scene.
# usage: bash scripts/gpu_r6_wide_blocks.sh <parent build> <kWideBlock 12 build> <kWideBlock 8 build> <output directory>
set -u
PARENT=$1; W12=$2; W8=$3; OUT=$4
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/gpu.csv" 2>&1; cat "$OUT/gpu.csv"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc $?"
python -m pytest -q tests/test_wide_tree_blocks.py tests/test_wide_tree.py tests/test_light_cull.py > "$OUT/pytest_wide.log" 2>&1; echo "wide/cull tests rc $?"
tail -3 "$OUT/pytest_wide.log"
BENCH="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline"
for i in 1 2 3; do
    $BENCH > "$OUT/w16_$i.json" 2> "$OUT/w16_$i.log"
    $BENCH --lib "$PARENT" > "$OUT/parent_$i.json" 2> "$OUT/parent_$i.log"
    $BENCH --lib "$W12" > "$OUT/w12_$i.json" 2> "$OUT/w12_$i.log"
    $BENCH --lib "$W8" > "$OUT/w8_$i.json" 2> "$OUT/w8_$i.log"
done
$BENCH --steps 3 --no-ref-work --dump-outputs "$OUT/dump_new" > /dev/null 2> "$OUT/dump_new.log"
$BENCH --steps 3 --no-ref-work --dump-outputs "$OUT/dump_old" --lib "$PARENT" > /dev/null 2> "$OUT/dump_old.log"
python - "$OUT" <<'PY'
import sys, numpy as np
out = sys.argv[1]
for f in ("frame.npy", "ray_counts.npy", "frame_pixels.npy"):
    a, b = np.load(f"{out}/dump_new/{f}"), np.load(f"{out}/dump_old/{f}")
    print(f, "identical" if a.shape == b.shape and np.array_equal(a, b) else "DIFFERENT")
PY
rm -rf "$OUT/dump_new" "$OUT/dump_old"
for t in w16 parent w12; do
    case $t in w16) L="";; parent) L="--lib $PARENT";; w12) L="--lib $W12";; esac
    RTB200_TRACE=1 $BENCH --steps 1 --no-ref-work $L > "$OUT/trace_$t.json" 2> "$OUT/trace_$t.log"
    echo "== $t"; grep -E "wide tree|packets .* histogram|split (shadow|primary)" "$OUT/trace_$t.log"
done
RTB200_TRACE=1 python - > /dev/null 2> "$OUT/nested_trace.log" <<'PY'
import sys
sys.path.insert(0, ".")
from tests import test_wide_tree_blocks as t
from raytracercpp_b200 import api
make, kw, where = t.SCENES["nested"]
t.render(api.load_library(), make(), kw, {}, **where)
PY
echo "== nested"; grep -E "wide tree" "$OUT/nested_trace.log"
python - "$OUT" <<'PY'
import glob, json, os, sys
out = sys.argv[1]
for f in sorted(glob.glob(f"{out}/*_[0-9].json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
    except Exception as e:
        print(os.path.basename(f), "no result", e); continue
    st = d["roofline"]["stage_ms_per_step"]
    print(f"{os.path.basename(f):20s} {d['ms_per_step']:8.3f} ms  primary {st['k_primary']:.3f} shade {st['k_shade']:.3f} "
          f"build {d['bvh']['build_ms']:.1f} ms  fetched p/s {d['work']['primary_fetched_bytes']}/{d['work']['shadow_fetched_bytes']}  "
          f"clock {d['clocks'].get('sm_mhz')}")
PY
