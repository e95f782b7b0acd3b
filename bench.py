#!/usr/bin/env python
"""bench.py -- Mrays/s (primary + shadow) of the ray-tracing hot path on BASELINE.json's headline configuration:
synthetic 10 M-triangle displaced sphere, 3840x2160, 16 spp (ssaa_factor 4), one point light with hard shadows,
screen-tile sharded over N GPUs (strong scaling: the frame is fixed, the tiles are dealt over the ranks).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU tracer (oracle/_ref) on the host cores
    python bench.py --dump-outputs DIR ...    # also writes what the last timed step computed (dump_outputs) as DIR/*.npy

A step is one full frame.  `value` = rays of the whole frame / device time (CUDA events on the launching stream, scene
and all buffers resident in HBM, max over ranks); `e2e` = the same frame through the public call with a HOST
framebuffer (camera/settings in, 33 MB ARGB32 out, copies inside the timed region).  One JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (triangles, width, height, ssaa, bvh_max_depth, bvh_leaf_object_count)
    "cfg4_sphere10M_4k_16spp": (10_000_000, 3840, 2160, 4, 12, 40),    # BASELINE.json configs[3]: the headline configuration (default)
    # the same mesh and frame with the camera 0.2 in front of the surface: 96 % of the samples hit, so traversal throughput is
    # not averaged with samples that never get a ray (cfg4 proper: the sphere covers 8 % of the frame)
    "cfg4_fill_sphere10M_4k_16spp": (10_000_000, 3840, 2160, 4, 12, 40),
    "sphere1M_1080p_4spp": (1_000_000, 1920, 1080, 2, 12, 40),         # for quick local checks only
    "cfg5_hair1M_4k": (1_000_000, 3840, 2160, 1, 12, 40),              # BASELINE.json configs[4]: ~1 M thin strand triangles, 4K, shadows
    # BASELINE.json configs[0..2] on the robot mesh (tests/golden/robot_scene.npz, cut from tp2/data/Robot/robot.obj)
    "cfg1_robot_720p": (3238, 1280, 720, 1, 12, 40),
    "cfg2_robot_textured_720p_4spp": (3238, 1280, 720, 2, 12, 40),
    "cfg3_robot_reflect16_1080p": (3238, 1920, 1080, 1, 12, 40),
}
FOV, LIGHT = 80.0, (3.0, 3.0, 2.0)
REFERENCE_BUILD = ("unmodified reference sources, g++ -O3 -mfma -fopenmp -march=x86-64-v3 (oracle/Makefile; the reference's own CMake uses "
                   "-march=native, which would not run on another host's CPU)")
CAMERA_Z = {"cfg4_fill_sphere10M_4k_16spp": -1.8}                       # camera_to_world = Translation(0, 0, z); identity elsewhere


def host_cpus() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Exactly ONE line may reach stdout: the JSON.  Libraries write there too (NCCL prints its version banner on stdout), so
# file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a private copy of the real stdout.
_JSON_OUT = None


def claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


# 24 B per dumped pixel (16 B of float32 channels in frame.npy + an 8 B float64 index in frame_pixels.npy): 48 MiB at most
DUMP_PIXELS = 1 << 21
RAY_COUNTERS = ("primary_rays", "shadow_rays", "reflection_rays", "reflection_shadow_rays", "primary_hits")


def dump_outputs(out_dir, argb, counts):
    """What the timed path handed its caller in the last timed step, for comparing two builds output for output (the
    inputs of a workload are seeded, so they are the same from run to run):
      frame.npy        [n, 4] float32: the A, R, G, B bytes of the ARGB32 frame at the pixels of frame_pixels.npy
      frame_pixels.npy [n] float64: their row-major indices -- every pixel, or a fixed seeded sample of DUMP_PIXELS of them
      ray_counts.npy   [5] float64: the step's RAY_COUNTERS summed over the ranks (the whole frame at any GPU count)"""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    argb = np.ascontiguousarray(argb).view(np.uint32).reshape(-1)
    idx = np.arange(argb.size)
    if argb.size > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(argb.size, DUMP_PIXELS, replace=False))
    px = argb[idx]
    np.save(out / "frame.npy", np.stack([(px >> np.uint32(s)) & np.uint32(0xff) for s in (24, 16, 8, 0)], -1).astype(np.float32))
    np.save(out / "frame_pixels.npy", idx.astype(np.float64))
    np.save(out / "ray_counts.npy", np.float64(counts))


def make_scene(name):
    from raytracercpp_b200 import scenes
    from raytracercpp_b200.renderer import precompute_materials
    tris, w, h, f, depth, leaf = WORKLOADS[name]
    kw = dict(image_width=w, image_height=h, enable_ssaa=int(f > 1), ssaa_factor=f, compute_shadows=1, bvh_max_depth=depth,
              bvh_leaf_object_count=leaf)
    tex = {}
    if "robot" in name:
        z = np.load(ROOT / "tests" / "golden" / "robot_scene.npz")
        xyz9, uv6, mat = z["xyz9"], z["uv6"], z["mat"]
        mats = [dict(ambient_coeff=tuple(r[0:3]), diffuse=tuple(r[3:6]), specular=tuple(r[6:9]), emission=tuple(r[9:12]),
                     reflection=float(r[12]), roughness=float(r[13]), ns=float(r[14]), specular_threshold=float(r[15])) for r in z["materials"]]
        if name.startswith("cfg2"):                        # 2048^2 u8 maps: AO, diffuse, normal (SURVEY.md 8(d) input 2)
            tex = {0: scenes.noise_texture((2048, 2048), 2), 1: scenes.noise_texture((2048, 2048), 1, "rgb"), 2: scenes.normal_map_texture((2048, 2048), 4)}
            kw.update(enable_ao_mapping=1, enable_diffuse_mapping=1, enable_normal_mapping=1)
        if name.startswith("cfg3"):                        # 16-ray rough fan, depth 1, roughness map, 4096x2048 sky (input 3)
            mats[0].update(reflection=0.9, roughness=0.0, specular=(0.2, 0.2, 0.2), diffuse=(0.5, 0.5, 0.5))
            mats[1].update(reflection=0.5, roughness=0.4)
            mats = precompute_materials(mats)
            tex = {3: scenes.noise_texture((2048, 2048), 3), 4: scenes.sky_texture((2048, 4096))}
            kw.update(rough_reflections_sample_count=16, max_recursion_depth=1, enable_roughness_mapping=1, enable_skysphere=1, rng_seed=7)
    else:
        if "hair" in name:
            xyz9, uv6, mat = scenes.hair_ball(n_strands=tris // 64, segments=16)
        else:
            xyz9, uv6, mat = scenes.displaced_sphere(*scenes.sphere_grid_for(tris))
        mats = precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
    cam = np.eye(4, dtype=np.float32)
    cam[2, 3] = CAMERA_Z.get(name, 0.0)
    return dict(xyz9=xyz9, uv6=uv6, mat=mat, mats=mats, kw=kw, name=name, tex=tex, cam=cam)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
def reference_sample(scene, row_step, threads=None, renderer=None, tracer=None):
    """Times the compiled reference (oracle/_ref/libref.so, or the oracle port if that was never built) on every
    `row_step`-th row of the supersampled frame, driving the reference's public trace_ray per pixel exactly as its
    ray_trace() loop does.  Returns (renderer, rays, ms, kind, cores)."""
    from oracle import bindings
    if tracer is None:
        kind = "reference" if bindings.available("ref") else "port"
        tracer = bindings.CpuTracer("ref" if kind == "reference" else "oracle")
    kind = "reference" if tracer.kind == "ref" else "port"
    # every host core this process may run on, stated explicitly: a launcher's OMP_NUM_THREADS (torchrun exports 1 for
    # every rank when nproc-per-node > 1) must not starve the CPU arm
    threads = host_cpus() if not threads or threads <= 0 else threads
    if renderer is None:
        s = bindings.default_settings(**scene["kw"])
        renderer = tracer.renderer()
        renderer.configure(s, FOV)
        t0 = time.time()
        renderer.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
        log(f"[reference] BVH::BVH over {len(scene['xyz9'])} triangles: {time.time() - t0:.1f} s")
        renderer.set_materials(scene["mats"])
        renderer.set_light(LIGHT)
        if not np.array_equal(scene["cam"], np.eye(4, dtype=np.float32)):
            renderer.set_camera_transform(scene["cam"])
        for slot, img in scene["tex"].items():
            renderer.set_texture(slot, img)
    rw, rh = renderer._super_dims()
    _, ms = renderer.trace_rows(row_begin=row_step // 2, row_end=rh, row_step=row_step, reseed=False, threads=threads, want_image=False)
    rows = len(range(row_step // 2, rh, row_step))
    if kind == "reference" and not scene["kw"].get("rough_reflections_sample_count"):
        rays = rows * rw + renderer.last_hit_count()
    else:
        # fan rays are not visible through the reference's public interface: counted (untimed) by the oracle port, whose
        # ray tree is the reference's (tests/test_oracle_vs_reference.py)
        counter = renderer if kind == "port" else scene.setdefault("_oracle_counter", _oracle_counter(scene))
        c = counter.count_rows(row_begin=row_step // 2, row_end=rh, row_step=row_step)
        rays = c["primary_rays"] + c["shadow_rays"] + c["reflection_rays"] + c["reflection_shadow_rays"]
    return renderer, tracer, rays, ms, kind, threads


def _oracle_counter(scene):
    from oracle import bindings
    r = bindings.CpuTracer("oracle").renderer()
    r.configure(bindings.default_settings(**scene["kw"]), FOV)
    r.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
    r.set_materials(scene["mats"])
    r.set_light(LIGHT)
    r.set_camera_transform(scene["cam"])
    for slot, img in scene["tex"].items():
        r.set_texture(slot, img)
    return r


def run_reference(args, scene):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle import bindings
    if not (bindings.available("ref") or bindings.available("oracle")):
        emit({"impl": "reference", "unavailable": "neither oracle/_ref/libref.so nor oracle/liboracle.so is built"})
        return
    kw = scene["kw"]
    rh = kw["image_height"] * kw["ssaa_factor"]
    # calibrate on a sparse sample, then size the per-step sample so that W + K steps take about two minutes
    renderer, tracer, rays, ms, kind, cores = reference_sample(scene, row_step=max(rh // 16, 1))
    per_ray_ms = ms / max(rays, 1)
    budget_ms = 120_000.0 / (args.steps + args.warmup)
    total_rays_est = rays * max(rh // 16, 1)
    row_step = int(max(1, np.ceil(total_rays_est * per_ray_ms / budget_ms)))
    log(f"[reference] calibration {ms:.0f} ms for {rays} rays -> row_step {row_step}")
    times, nrays = [], 0
    for i in range(args.warmup + args.steps):
        _, _, rays, ms, _, _ = reference_sample(scene, row_step, renderer=renderer, tracer=tracer)
        if i >= args.warmup:
            times.append(ms)
            nrays = rays
    ms_step = float(np.mean(times))
    value = nrays / ms_step / 1e3
    sample = f"every {row_step}th row of the {kw['image_width'] * kw['ssaa_factor']}x{rh} supersampled frame ({nrays} rays per step)"
    out = {
        "impl": "reference", "metric": "Mrays/s (primary+shadow)", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(scene, args.gpus, args.tile),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample,
                         "build": REFERENCE_BUILD if kind == "reference" else "oracle/oracle.cpp (port)"},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


def workload_config(scene, n_gpus, tile=64):
    kw = scene["kw"]
    return {"workload": scene["name"], "triangles": int(len(scene["xyz9"])), "image": f"{kw['image_width']}x{kw['image_height']}",
            "spp": kw["ssaa_factor"] ** 2, "primary_rays": kw["image_width"] * kw["image_height"] * kw["ssaa_factor"] ** 2,
            "shadows": "1 point light, hard", "bvh": f"octree max_depth {kw['bvh_max_depth']} leaf {kw['bvh_leaf_object_count']} (reference GUI defaults)",
            "fov": FOV, "parallelism": f"screen tiles {tile}x{tile} round-robin over {n_gpus} GPU(s), scene replicated",
            "l2": "scene (~0.9 GB) and sample buffer (0.5 GB) exceed the 126 MB L2; no flush between steps"}


# ---------------------------------------------------------------------------------------------------------------
def setup_context(ctx, api, scene, args, leaf_split=None):
    kw = scene["kw"]
    if leaf_split is not None:
        ctx.set_option(api.RT_OPT_LEAF_SPLIT, leaf_split)
    for kv in args.opt:
        k, v = kv.split("=")
        ctx.set_option(int(k), int(v))
    info = ctx.build_bvh(kw["bvh_max_depth"], kw["bvh_leaf_object_count"])
    ctx.set_materials(scene["mats"])
    ctx.set_light(LIGHT)
    for slot, img in scene["tex"].items():
        ctx.set_texture(slot, img)
    f = kw["ssaa_factor"] if kw["enable_ssaa"] else 1
    aspect = float(np.float32(kw["image_width"] * f) / np.float32(kw["image_height"] * f))
    proj_inv = ctx.perspective_inverse(FOV, aspect)
    cam = scene["cam"]
    pos = ctx.transform_point(cam, (0, 0, 0))
    ctx.set_camera(proj_inv, cam, pos)
    return info, (proj_inv, cam, pos)


def run_ours(args, scene):
    import torch
    import torch.distributed as dist
    from raytracercpp_b200 import api
    from raytracercpp_b200.distributed import FramePipeline, ShardedFrame

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = api.load_library(args.lib)
    # host threads of the library's own loops (octree build, copy into the caller's frame): this rank's share of the
    # box's cores, whatever OMP_NUM_THREADS the launcher exported (torchrun: 1)
    host_threads = max(1, host_cpus() // max(local_world, 1))
    lib.rt_set_host_threads(host_threads)
    ctx = api.Context(local, lib)
    kw = scene["kw"]
    s = api.default_settings(lib, **kw)
    ctx.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
    lanes_on = not any(kv.split("=")[0] == str(api.RT_OPT_LANES) and int(kv.split("=")[1]) == 0 for kv in args.opt)
    graph_on = not any(kv.split("=")[0] == str(api.RT_OPT_GRAPH) and int(kv.split("=")[1]) == 0 for kv in args.opt)
    ref_work = None
    if not args.no_ref_work:
        # Work of the REFERENCE-SHAPED traversal (SURVEY.md section 8(d)): the reference's own cells and leaves
        # (RT_OPT_LEAF_SPLIT 0), one ordered early-exit traversal per ray (RT_OPT_PACKETS 0), instrumented kernels.
        # Outside every timed region; the product tree is built afterwards.
        setup_context(ctx, api, scene, args, leaf_split=0)
        ctx.set_option(api.RT_OPT_PACKETS, 0)
        ctx.set_option(api.RT_OPT_COUNT_WORK, 1)
        ref_frame = ShardedFrame(ctx, s, rank, world, tile_size=args.tile, gather="nccl")
        ref_work = ref_frame.render().as_dict()
        del ref_frame
        ctx.set_option(api.RT_OPT_COUNT_WORK, 0)
        ctx.set_option(api.RT_OPT_PACKETS, 1)
        if rank == 0:
            log(f"[ours] reference-shaped traversal: {ref_work['primary_volume_tests']} + {ref_work['shadow_volume_tests']} volume tests, "
                f"{ref_work['primary_triangle_tests']} + {ref_work['shadow_triangle_tests']} triangle tests (primary + shadow)")
    info, (proj_inv, cam, pos) = setup_context(ctx, api, scene, args, leaf_split=args.leaf_split if args.leaf_split is not None else 8)
    if rank == 0:
        log(f"[ours] octree build {info['build_ms']:.0f} ms ({host_threads} host threads) + upload {info['upload_ms']:.0f} ms, "
            f"{info['child_records']} records, {info['device_bytes'] / 1e6:.0f} MB resident, max leaf {info['max_leaf_size']}")
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    frame = ShardedFrame(ctx, s, rank, world, tile_size=args.tile, gather=args.gather)
    if rank == 0 and world > 1:
        log(f"[ours] frame gather mode: {frame.mode}" + (f" (peer refused: {frame.why_not_peer})" if frame.why_not_peer else ""))

    # More frames in flight (--frames-in-flight F, default 2): F - 1 further contexts with the same scene, each on its own
    # stream with its own frame buffers; the timed loop enqueues frame k+1 before it waits for frame k (FramePipeline).
    # default: 2 on one or two GPUs, 1 on more -- measured on the 8-GPU box: 2.53 ms per frame with one frame at a time, 3.16 ms
    # with two (two frames' kernels side by side spread the ranks' finishing times, and every frame waits at its barrier for
    # the slowest rank); on 1 / 2 GPUs two in flight gain 2 %
    in_flight = args.frames_in_flight if args.frames_in_flight > 0 else (2 if world <= 2 else 1)
    frames, streams, ctxs = [frame], [stream], [ctx]
    for _ in range(1, in_flight):
        c2 = api.Context(local, lib)
        c2.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
        setup_context(c2, api, scene, args, leaf_split=args.leaf_split if args.leaf_split is not None else 8)
        st2 = torch.cuda.Stream()
        c2.set_stream(st2.cuda_stream)
        ctxs.append(c2); streams.append(st2)
        frames.append(ShardedFrame(c2, s, rank, world, tile_size=args.tile, gather=args.gather))
    pipe = FramePipeline(frames, streams)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # --- work of the traversal (instrumented instantiations, outside every timed region)
    ctx.set_option(api.RT_OPT_COUNT_WORK, 1)
    with torch.cuda.stream(stream):
        work = frame.render()
    ctx.set_option(api.RT_OPT_COUNT_WORK, 0)

    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 2 * in_flight)):                          # every context warms up (and captures its frame graphs)
            pipe.submit()
        pipe.drain()
        sync_all()
        sampler = ClockSampler(local)
        sampler.start()
        stage = {"k_primary": 0.0, "k_compact": 0.0, "k_shade": 0.0, "k_reflect": 0.0, "k_resolve": 0.0}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        st = None
        # the timed region starts on every stream at ev0 and ends when the last stream is done: K frames, F in flight
        ev0.record(stream)
        for other in streams[1:]:
            other.wait_event(ev0)
        done = []
        for _ in range(args.steps):
            r = pipe.submit()
            if r is not None:
                done.append(r)
        done += pipe.drain()
        for other in streams[1:]:
            e = torch.cuda.Event()
            e.record(other)
            stream.wait_event(e)
        ev1.record(stream)
        sync_all()
        assert len(done) == args.steps
        st = done[-1]
        # --dump-outputs: a device copy of the last timed frame (its buffer is rendered into again below); it goes to the
        # host and to disk only after every measurement
        last_frame = frames[(pipe.next - 1) % len(frames)].frame.clone() if args.dump_outputs and rank == 0 else None
        last_counts = [getattr(st, k) for k in RAY_COUNTERS]
        launches = sum(d.kernel_launches + (2 if frame.mode == "nccl" else 0) for d in done)   # + the pack and unpack kernels of the nccl-mode gather
        dev_ms = ev0.elapsed_time(ev1)
        rays_rank, traced_rank = st.total_rays, st.traced_rays
        # Per-kernel durations for the roofline: the SAME K frames once more, still inside the clock sampling, with the two
        # chunk lanes turned off (RT_OPT_LANES 0) -- with two lanes the kernels of the two chunks overlap on purpose and a
        # CUDA-event pair around one of them also measures the time it waits for SMs.
        ctx.set_option(api.RT_OPT_LANES, 0)
        ctx.set_option(api.RT_OPT_GRAPH, 0)                                       # a replayed frame graph has no per-stage events
        serial0, serial1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        frame.render_and_gather()
        serial0.record(stream)
        for _ in range(args.steps):
            st = frame.render_and_gather()
            stage["k_primary"] += st.trace_primary_ms; stage["k_shade"] += st.shade_ms
            stage["k_reflect"] += st.reflect_ms; stage["k_resolve"] += st.resolve_ms; stage["k_compact"] += st.compact_ms
        serial1.record(stream)
        sync_all()
        serial_ms = serial0.elapsed_time(serial1) / args.steps
        ctx.set_option(api.RT_OPT_LANES, 1 if lanes_on else 0)
        ctx.set_option(api.RT_OPT_GRAPH, 1 if graph_on else 0)
        clocks = sampler.stop()

        # --- end to end through the public call: the frame ends up in an ordinary (pageable) host array of the caller.
        # N = 1: rt_render(ctx, settings, argb_out).  N > 1: the sharded counterpart (ShardedFrame.render_to_host: every rank
        # renders its tiles into rank 0's frame, rank 0 copies it out with rt_frame_to_host).  Inputs of a step: camera and
        # settings (host structs -> kernel arguments); result: the ARGB32 frame.  All copies are inside the timed region.
        host = np.empty((kw["image_height"], kw["image_width"]), np.uint32)
        host.fill(0)                                                             # touch the pages once, as a GUI's frame buffer would be

        e2e_device_ms = []

        def e2e_step():
            ctx.set_camera(proj_inv, cam, pos)
            if world == 1:
                e2e_device_ms.append(ctx.render(s, host)[1].device_ms)
            else:
                frame.render_to_host(host)

        for _ in range(min(args.warmup, 3)):
            e2e_step()
        sync_all()
        e2e_steps_ms = []
        t_e2e = time.perf_counter()
        for _ in range(args.steps):
            t_step = time.perf_counter()
            e2e_step()
            e2e_steps_ms.append((time.perf_counter() - t_step) * 1e3)
        stream.synchronize()
        e2e_ms = (time.perf_counter() - t_e2e) * 1e3
        log("[ours] e2e steps (ms): " + " ".join(f"{x:.2f}" for x in e2e_steps_ms) + " | device part: " + " ".join(f"{x:.2f}" for x in e2e_device_ms[-args.steps:]))

    # --- the frame of the sharded run must be the 1-GPU frame, on the device and in the caller's host array
    # (rank 0 renders every tile once more, untimed)
    frame_check = None
    if world > 1:
        with torch.cuda.stream(stream):
            frame.render_and_gather()
            stream.synchronize()
            if rank == 0:
                gathered = frame.frame.clone()
                whole = ShardedFrame(ctx, s, 0, 1, tile_size=args.tile)
                whole.render()
                stream.synchronize()
                same = bool(torch.equal(whole.frame, gathered)) and bool(np.array_equal(host, whole.frame.cpu().numpy().view(np.uint32)))
                frame_check = "identical to the 1-GPU frame (device frame and host array)" if same else "DIFFERS from the 1-GPU frame"
                if not same:
                    raise SystemExit("bench.py: the gathered frame differs from the 1-GPU frame")

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    mine = torch.tensor([stage[k] / args.steps for k in ("k_primary", "k_compact", "k_shade", "k_reflect", "k_resolve")] + [dev_ms / args.steps],
                        dtype=torch.float64, device="cuda")
    per_rank = [mine.tolist()]
    if world > 1:
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [[round(x, 3) for x in t.tolist()] for t in allr]
    dev_ms = reduce(dev_ms, dist.ReduceOp.MAX if world > 1 else None)
    e2e_ms = reduce(e2e_ms, dist.ReduceOp.MAX if world > 1 else None)
    rays_total = reduce(float(rays_rank), dist.ReduceOp.SUM if world > 1 else None)
    traced_total = reduce(float(traced_rank), dist.ReduceOp.SUM if world > 1 else None)
    launches_total = reduce(float(launches), dist.ReduceOp.SUM if world > 1 else None)
    if args.dump_outputs:
        counts = [reduce(float(c), dist.ReduceOp.SUM if world > 1 else None) for c in last_counts]
        if rank == 0:
            dump_outputs(args.dump_outputs, last_frame.cpu().numpy(), counts)
    ms_step = dev_ms / args.steps
    value = rays_total / ms_step / 1e3

    if rank == 0:
        peaks_file = ROOT / "MEASURED_PEAKS.json"
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        if peaks_file.exists():
            peak, peak_src = float(json.loads(peaks_file.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        dom = max(("k_primary", "k_shade", "k_reflect"), key=lambda k: stage[k])
        own = work.as_dict()
        pre = {"k_primary": "primary", "k_shade": "shadow", "k_reflect": "reflection"}[dom]
        fetched = own[pre + "_fetched_bytes"]                                     # rank 0's tiles, one launch set (= one step)
        dom_ms = stage[dom] / args.steps
        achieved = fetched / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        ref_bytes = None if ref_work is None else 56 * ref_work[pre + "_volume_tests"] + 36 * ref_work[pre + "_triangle_tests"]
        # ncu figures of the SAME kernel set, from the committed capture of this workload at N = 1 (scripts/make_profiles.py
        # writes profiles/traffic.json from the .ncu-rep; it names the commit it was taken at).  At N > 1 the launch covers
        # another set of tiles, so nothing is quoted there.
        prof = {}
        tf = ROOT / "profiles" / "traffic.json"
        if tf.exists() and world == 1:
            prof = json.loads(tf.read_text()).get(scene["name"], {}).get(dom, {})
            if not isinstance(prof, dict):
                prof = {}
        traffic = prof.get("dram_bytes")
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        n_sm = torch.cuda.get_device_properties(local).multi_processor_count
        issue_peak = n_sm * 4 * sm_mhz * 1e6                                      # warp instructions per second: 4 schedulers per SM, 1 per clock
        warp_inst = prof.get("warp_inst")
        issue = None
        if warp_inst and dom_ms > 0:
            issue = {"bound": "issue", "kernel": dom, "achieved": warp_inst / (dom_ms * 1e-3) / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-inst/s",
                     "frac": warp_inst / (dom_ms * 1e-3) / issue_peak, "warp_inst_per_launch": warp_inst,
                     "warp_inst_per_traced_ray": warp_inst / max(1, {"k_primary": st.traced_primary_rays, "k_shade": st.shadow_rays,
                                                                   "k_reflect": st.reflection_rays + st.reflection_shadow_rays}[dom]),
                     "source": prof.get("source"), "peak_definition": f"{n_sm} SMs x 4 schedulers x {sm_mhz:.0f} MHz (median SM clock of the timed region)"}
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "algorithmic_bytes_per_launch": fetched, "kernel_ms_per_step": dom_ms,
                    "definition": ("node + triangle bytes the kernel FETCHES per launch: 64 B per child record and 48 B per triangle, once per warp "
                                   "and test (a 32-ray packet shares each fetch), counted by the instrumented instantiation of the same kernels "
                                   "(RT_OPT_COUNT_WORK) outside the timed region; divided by the kernel's CUDA-event time in the timed run. "
                                   "`traffic` = DRAM bytes of the same launch set under ncu (the rest is served by the 126 MB L2). "
                                   "The kernel is ISSUE-bound, not HBM-bound: see roofline_issue"),
                    "dram_frac": (traffic / (dom_ms * 1e-3) / 1e9 / peak) if (traffic and dom_ms > 0) else None,
                    "reference_shaped_bytes": ref_bytes,
                    "reference_shaped_definition": "SURVEY.md 8(d): 56 B per volume test + 36 B per triangle test of one ordered early-exit traversal per "
                                                   "ray over the reference's own cells and leaves; a property of the reference algorithm, not bytes this kernel moves",
                    "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
                    "stage_timing": "K more frames with RT_OPT_LANES 0 (the chunks' kernels back to back on one stream; with the two lanes of "
                                    "the timed run they overlap on purpose), %.3f ms per frame that way" % serial_ms}
        cfg = workload_config(scene, world, args.tile)
        cfg["frames_in_flight"] = (f"{in_flight}: frame k+1 is enqueued (own context, stream and frame buffers) before the host waits for frame k; "
                                   "`ms_per_step` = time of the K frames / K" if in_flight > 1 else "1: each frame is waited for before the next is enqueued")
        cfg["gather"] = {"peer": "every rank's resolve kernel stores its tiles into rank 0's frame over NVLink (CUDA IPC), one 4-byte all-reduce per frame as the barrier",
                         "nccl": "pack kernel -> all_gather_into_tensor -> unpack kernel", "single": "none (one GPU)"}[frame.mode]
        out = {
            "metric": "Mrays/s (primary+shadow)", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "rays_per_step": int(rays_total), "traced_rays_per_step": int(traced_total),
            "traced_mrays_s": traced_total / ms_step / 1e3,
            "rays_note": ("`value` counts every sample of the frame plus the shadow (and fan) rays, as the reference arm does for the same frame; "
                          "`traced_*` leaves out the primary samples that the screen-space bound of the scene writes as misses without a ray"),
            "clocks": clocks,
            "e2e": {"value": rays_total / (e2e_ms / args.steps) / 1e3, "unit": "Mrays/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": 2 * 64 + 12 + 12 + 108, "d2h_bytes_per_step": int(host.size * 4),
                    "call": "rt_render into a pageable host array" if world == 1 else
                            "ShardedFrame.render_to_host: rt_render_device_begin on every rank (stores into rank 0's frame), barrier, rt_frame_to_host into a pageable host array on rank 0"},
            "gpu_launches": int(launches_total), "roofline": roofline, "roofline_issue": issue,
            "work": {k: own[k] for k in ("primary_volume_tests", "primary_triangle_tests", "shadow_volume_tests", "shadow_triangle_tests",
                                         "primary_hits", "primary_fetched_bytes", "shadow_fetched_bytes", "reflection_fetched_bytes")},
            "reference_work": None if ref_work is None else {k: ref_work[k] for k in ("primary_volume_tests", "primary_triangle_tests",
                                                                                      "shadow_volume_tests", "shadow_triangle_tests")},
            "per_rank_stage_ms": per_rank, "frame_check": frame_check,
            "bvh": dict({k: info[k] for k in ("nodes", "interior", "leaves", "empty_leaves", "max_leaf_size", "child_records", "device_bytes", "build_ms", "upload_ms")},
                        host_threads=host_threads),
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                _, _, rays, ms, kind, cores = reference_sample(scene, row_step=args.cpu_row_step)
                out["cpu_baseline"] = {"value": rays / ms / 1e3, "unit": "Mrays/s", "cores": cores, "kind": kind,
                                       "build": REFERENCE_BUILD if kind == "reference" else "oracle/oracle.cpp (port)",
                                       "sample": f"every {args.cpu_row_step}th row of the supersampled frame, {rays} rays in {ms / 1e3:.1f} s"}
            except Exception as e:  # the checker is optional for the GPU number, never the other way round
                out["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}
        emit(out)
    for f in frames:
        f.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4_sphere10M_4k_16spp", choices=list(WORKLOADS))
    ap.add_argument("--frames-in-flight", type=int, default=0,
                    help="frames enqueued before the host waits for the oldest (each on its own context and stream); 1 = one frame at a time; "
                         "0 (default) = 2 on one or two GPUs, 1 on more")
    ap.add_argument("--cpu-row-step", type=int, default=6, help="cpu_baseline sample: every n-th supersampled row")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-work", action="store_true", help="skip the reference-shaped work count (roofline then uses the kernel's own tests)")
    ap.add_argument("--opt", action="append", default=[], help="library option override id=value (experiments), e.g. --opt 3=4")
    ap.add_argument("--tile", type=int, default=None, help="side of the screen tiles dealt over the ranks (final-resolution pixels); "
                    "default 64 on one GPU, 32 on several (finer interleaving balances the ranks better, measured at N=8)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: how the frame gets to rank 0 (raytracercpp_b200/distributed.py)")
    ap.add_argument("--lib", default=None, help="another build of librtb200 (kernel A/B experiments)")
    ap.add_argument("--leaf-split", type=int, default=None, help="RT_OPT_LEAF_SPLIT override (experiments); default = library default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame and ray counters of the last timed step as DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    claim_stdout()
    if args.tile is None:
        args.tile = 64 if int(os.environ.get("WORLD_SIZE", 1)) == 1 else 32
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference" and int(os.environ.get("RANK", 0)) != 0:
        return
    t0 = time.time()
    scene = make_scene(args.workload)
    log(f"[{args.impl}] scene {args.workload}: {len(scene['xyz9'])} triangles generated in {time.time() - t0:.1f} s")
    if args.impl == "reference":
        run_reference(args, scene)
    else:
        run_ours(args, scene)


if __name__ == "__main__":
    main()
