"""bench.py --dump-outputs: what the timed path computed in its last step, as float .npy files (at most 64 MB)."""
import json
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def words(out):
    """The ARGB32 words back from frame.npy, and the pixels they belong to."""
    ch = np.load(out / "frame.npy").astype(np.uint32)
    return (ch[:, 0] << 24) | (ch[:, 1] << 16) | (ch[:, 2] << 8) | ch[:, 3], np.load(out / "frame_pixels.npy").astype(np.int64)


def test_dump_of_a_4k_frame_is_a_fixed_sample_under_64_mb(tmp_path):
    frame = np.random.default_rng(5).integers(0, 2**32, size=(2160, 3840), dtype=np.uint64).astype(np.uint32)
    counts = [1.0, 2.0, 3.0, 4.0, 5.0]
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, frame.view(np.int32), counts)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["frame.npy", "frame_pixels.npy", "ray_counts.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64e6
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)       # the same pixels every run
    w, idx = words(tmp_path / "a")
    assert len(idx) == bench.DUMP_PIXELS and len(np.unique(idx)) == len(idx)
    assert np.array_equal(w, frame.reshape(-1)[idx])
    assert np.load(tmp_path / "a" / "ray_counts.npy").tolist() == counts


def test_dump_of_a_small_frame_has_every_pixel(tmp_path):
    frame = np.arange(54 * 96, dtype=np.uint32).reshape(54, 96) * np.uint32(2654435761)
    bench.dump_outputs(tmp_path, frame, [0] * 5)
    w, idx = words(tmp_path)
    assert np.array_equal(idx, np.arange(frame.size)) and np.array_equal(w, frame.reshape(-1))


@pytest.mark.gpu
def test_bench_dump_is_the_rendered_frame(cuda_lib, tmp_path):
    """The dump of a bench run is the frame (and ray counts) that rt_render gives for the same workload and settings."""
    name = "cfg1_robot_720p"
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", name, "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--no-ref-work", "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert p.returncode == 0, p.stderr[-3000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
    from raytracercpp_b200 import api
    scene = bench.make_scene(name)
    ctx = api.Context(0, cuda_lib)
    ctx.set_triangles(scene["xyz9"], scene["uv6"], scene["mat"])
    bench.setup_context(ctx, api, scene, types.SimpleNamespace(opt=[]), leaf_split=8)
    want, stats = ctx.render(api.default_settings(cuda_lib, **scene["kw"]))
    w, idx = words(tmp_path / "out")
    assert len(idx) == want.size                                               # 1280 x 720 is under DUMP_PIXELS: every pixel
    assert np.array_equal(w, want.reshape(-1)[idx])
    assert np.load(tmp_path / "out" / "ray_counts.npy").tolist() == [float(getattr(stats, k)) for k in bench.RAY_COUNTERS]
    ctx.close()
