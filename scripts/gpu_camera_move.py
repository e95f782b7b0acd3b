"""Cost of moving the camera on bench.py's headline scene (10 M-triangle sphere, 4K, 16 spp, one GPU): the screen coverage of
the primary packets (rtb200.cu: screen_coverage) is rebuilt on the host and uploaded at the first frame after a move, the
tile split is redone, and that frame cannot replay a captured frame graph.  Prints one JSON line: steady frames, the three
frames after a move (ordinary enqueue with the rebuild, capture, replay), and frames whose camera moves every time, with the
cull on and off.  Times are the frames' CUDA-event times (RtRenderStats.device_ms) and host wall times around rt_render
(which ends in a device synchronise).  With RTB200_TRACE=1 the library also prints the rebuild and the upload on their own
("[rtb200] screen coverage ...").
usage: python scripts/gpu_camera_move.py [--lib other/librtb200.so] [--moves N]"""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
from raytracercpp_b200 import api  # noqa: E402


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
    _, (pinv, cam0, _) = bench.setup_context(ctx, api, scene, argparse.Namespace(opt=[]))

    def pose(i):
        """bench's camera, or that camera shifted and turned a little (the sphere stays on screen)"""
        m = np.asarray(cam0, np.float32).reshape(4, 4).copy()
        if i % 2:
            a = 0.03
            turn = np.float32([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
            m[:3, :3] = m[:3, :3] @ turn
            m[:3, 3] += np.float32([0.05, -0.03, 0.02])
        return m

    def frame(i=None):
        if i is not None:
            m = pose(i)
            ctx.set_camera(pinv, m, ctx.transform_point(m, (0, 0, 0)))
        t0 = time.perf_counter()
        st = ctx.render(s)[1]
        return st.device_ms, 1e3 * (time.perf_counter() - t0)

    frame(0)
    out = {"triangles": int(len(scene["xyz9"]))}
    for _ in range(4):
        frame()
    steady = [frame() for _ in range(10)]
    out["steady_ms"] = {"device": statistics.median(f[0] for f in steady), "host": statistics.median(f[1] for f in steady)}
    after = []
    for i in range(args.moves):
        after.append([frame(i + 1), frame(), frame()])
    out["after_move_ms"] = {k: {"device": statistics.median(a[j][0] for a in after), "host": statistics.median(a[j][1] for a in after)}
                            for j, k in enumerate(("first", "second_capture", "third_replay"))}
    for cull in (1, 0):
        ctx.set_option(api.RT_OPT_SCREEN_CULL, cull)
        frame(0); frame()
        every = [frame(i + 1) for i in range(2 * args.moves)]
        out[f"camera_moves_every_frame_cull{cull}_ms"] = {"device": statistics.median(f[0] for f in every),
                                                          "host": statistics.median(f[1] for f in every)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
