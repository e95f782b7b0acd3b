"""Where each frame's slab and triangle tests go: one rt_render_work_map frame of each of bench.py's cfg4 (10 M-triangle sphere,
4K, 16 spp), cfg4_fill (the same with the camera in front of the surface), cfg5 (1 M hair triangles, 4K) and cfg3 (robot, 1080p,
16-ray rough reflection fans), at their bench sizes and with the library's default options.

Writes <out>/work_map.json: per workload and ray class (primary, shadow, reflection), the totals of the map against the frame's
RtRenderStats counters, the volume / triangle tests per pixel (mean, p50, p99, max), and the share of the class's work
(56 B per volume test + 36 B per triangle test, the bytes-per-ray metric of DESIGN.md) that lies in the costliest 1 % and
10 % of pixels.  And <maps>/<workload>_<class>.pgm: that work summed over 8x8-pixel cells (1/8 resolution), log-scaled to
8 bits, top row first.  The time it records is the CUDA-event time of the INSTRUMENTED frame (the counting kernels, plus the
per-pixel atomics), never a timed frame; the card's name and power limit are read in the same run and stored beside it.
usage: python scripts/gpu_work_map.py [--out profiles] [--maps build/work_map] [--lib other/librtb200.so] [--workloads a,b]"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
from raytracercpp_b200 import api  # noqa: E402

WORKLOADS = ["cfg4_sphere10M_4k_16spp", "cfg4_fill_sphere10M_4k_16spp", "cfg5_hair1M_4k", "cfg3_robot_reflect16_1080p"]
CLASSES = ("primary", "shadow", "reflection")


def card():
    """name, power limit and max SM clock of GPU 0 (nvidia-smi), read in the same run as the frames"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                                   # the numbers below then stand without a card
        return {"error": f"nvidia-smi: {e}"}


def per_pixel(x):
    x = x.astype(np.float64).ravel()
    return {"mean": float(x.mean()), "p50": float(np.percentile(x, 50)), "p99": float(np.percentile(x, 99)), "max": float(x.max())}


def top_share(cost, frac):
    """share of the sum of `cost` held by the ceil(frac * n) largest entries"""
    c = cost.ravel()
    total = float(c.sum())
    if total == 0.0:
        return 0.0
    k = max(1, int(np.ceil(frac * c.size)))
    return float(np.partition(c, c.size - k)[c.size - k:].sum()) / total


def write_pgm(path, cost):
    """log-scaled 8-bit heat map of `cost` summed over 8x8-pixel cells; rows flipped so that the top row comes first"""
    h, w = cost.shape
    hh, ww = (h + 7) // 8, (w + 7) // 8
    pad = np.zeros((hh * 8, ww * 8), np.float64)
    pad[:h, :w] = cost
    cells = pad.reshape(hh, 8, ww, 8).sum(axis=(1, 3))[::-1]
    top = np.log1p(cells.max()) if cells.max() > 0 else 1.0
    img = np.round(255.0 * np.log1p(cells) / top).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (ww, hh))
        f.write(img.tobytes())


def measure(lib, name, maps_dir):
    scene = bench.make_scene(name)
    ctx = api.Context(0, lib)
    try:
        s = api.default_settings(lib, **scene["kw"])
        ctx.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
        bench.setup_context(ctx, api, scene, argparse.Namespace(opt=[]))
        ctx.render_work_map(s)                                               # first call: allocations, module loads
        _, work, st = ctx.render_work_map(s)
    finally:
        ctx.close()
    out = {"image": [s.image_width, s.image_height], "ssaa_factor": s.ssaa_factor if s.enable_ssaa else 1,
           "instrumented_frame_device_ms": st.device_ms,
           "rays": {k: getattr(st, k) for k in ("primary_rays", "traced_primary_rays", "shadow_rays", "reflection_rays", "reflection_shadow_rays")},
           "classes": {}}
    for cls in CLASSES:
        v, t = work[f"{cls}_volume_tests"], work[f"{cls}_triangle_tests"]
        sv, stt = int(v.sum(dtype=np.uint64)), int(t.sum(dtype=np.uint64))
        cost = 56.0 * v.astype(np.float64) + 36.0 * t.astype(np.float64)
        out["classes"][cls] = {
            "volume_tests": sv, "triangle_tests": stt,
            "equals_stats": sv == getattr(st, f"{cls}_volume_tests") and stt == getattr(st, f"{cls}_triangle_tests"),
            "volume_tests_per_pixel": per_pixel(v), "triangle_tests_per_pixel": per_pixel(t),
            "pixels_with_work": int((cost > 0).sum()),
            "share_in_costliest_1pct_pixels": top_share(cost, 0.01), "share_in_costliest_10pct_pixels": top_share(cost, 0.10),
        }
        if maps_dir is not None:
            write_pgm(maps_dir / f"{name}_{cls}.pgm", cost)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--maps", default=str(ROOT / "build" / "work_map"), help="directory of the PGM heat maps ('' = none)")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    lib = api.load_library(args.lib)
    maps_dir = Path(args.maps) if args.maps else None
    if maps_dir is not None:
        maps_dir.mkdir(parents=True, exist_ok=True)
    result = {"what": "per-pixel traversal work (rt_render_work_map) of one frame per workload, default options; times are of the "
                      "instrumented frame, not a timed one", "card": card(), "workloads": {}}
    for name in args.workloads.split(","):
        result["workloads"][name] = measure(lib, name, maps_dir)
        r = result["workloads"][name]
        print(name, "instrumented frame %.2f ms" % r["instrumented_frame_device_ms"],
              " ".join(f"{c}: V {r['classes'][c]['volume_tests']} T {r['classes'][c]['triangle_tests']} "
                       f"top1% {r['classes'][c]['share_in_costliest_1pct_pixels']:.3f} ok={r['classes'][c]['equals_stats']}" for c in CLASSES), flush=True)
    Path(args.out).mkdir(parents=True, exist_ok=True)
    (Path(args.out) / "work_map.json").write_text(json.dumps(result, indent=1) + "\n")
    ok = all(c["equals_stats"] for w in result["workloads"].values() for c in w["classes"].values())
    print("card:", result["card"], "| map totals equal the stats:", ok)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
