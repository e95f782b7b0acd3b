"""Cost of moving the point light on bench.py's headline scene (10 M-triangle sphere, 4K, 16 spp, one GPU): the light-cull
masks (csrc/light_cull.cuh) are rebuilt at the first frame after a move, and that frame cannot replay a captured frame graph.
Prints one JSON line: the octree build, steady frames, the three frames after a move (ordinary enqueue with the mask
rebuild, capture, replay), and frames whose light moves every time, with the cull on and off.  Device times are the
frames' CUDA-event times (RtRenderStats.device_ms, which include the mask rebuild).  With RTB200_TRACE=1 the library
also prints the mask pass on its own ("[rtb200] light_mask ... ms", CUDA events around its launches).
usage: python scripts/gpu_light_move.py [--lib other/librtb200.so] [--moves N]"""
import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
from raytracercpp_b200 import api  # noqa: E402

LIGHT2 = (2.5, 3.2, 1.5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--moves", type=int, default=8)
    args = ap.parse_args()
    scene = bench.make_scene("cfg4_sphere10M_4k_16spp")
    lib = api.load_library(args.lib)
    ctx = api.Context(0, lib)
    s = api.default_settings(lib, **scene["kw"])
    ctx.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
    info, _ = bench.setup_context(ctx, api, scene, argparse.Namespace(opt=[]))
    rebuilt = [ctx.build_bvh(scene["kw"]["bvh_max_depth"], scene["kw"]["bvh_leaf_object_count"])["build_ms"] for _ in range(3)]

    def frame(light=None):
        if light is not None:
            ctx.set_light(light)
        return ctx.render(s)[1].device_ms

    out = {"triangles": int(len(scene["xyz9"])), "octree_build_ms": rebuilt}
    for _ in range(4):
        frame()
    out["steady_ms"] = statistics.median(frame() for _ in range(10))
    after = []
    for i in range(args.moves):
        light = LIGHT2 if i % 2 == 0 else bench.LIGHT
        after.append([frame(light), frame(), frame()])
    out["after_move_ms"] = {k: statistics.median(a[j] for a in after) for j, k in enumerate(("first", "second_capture", "third_replay"))}
    for cull in (1, 0):
        ctx.set_option(api.RT_OPT_LIGHT_CULL, cull)
        frame(); frame()
        every = [frame(LIGHT2 if i % 2 == 0 else bench.LIGHT) for i in range(2 * args.moves)]
        out[f"light_moves_every_frame_cull{cull}_ms"] = statistics.median(every)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
