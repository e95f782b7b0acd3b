"""Cuts tests/golden/golden_raster.npz: frames of Renderer::raster_trace() + post_process() (hybrid_rasterization_tracing,
renderer.cpp:869-1006) from the UNMODIFIED reference compiled in this container (oracle/_ref/libref_strict.so), run on ONE
thread -- raster_trace() walks the triangles under `omp parallel for` over an unsynchronised z-buffer, so the sequential
order is the reproducible one -- and, for the SSAO case, after srand(RASTER_SRAND) as in make_golden_ssao.py.

    python tests/golden/make_golden_raster.py        (needs the original sources: RTB200_REFERENCE, see make_golden.py)

Per set-up of tests/common.py::raster_table that has no rough reflections: the reference's frame (and the nine SSAO
generator seeds where SSAO is on).  The oracle must reproduce every frame bit for bit before the file is written.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.bindings import CpuTracer  # noqa: E402
from tests.conftest import require_reference  # noqa: E402
from tests import common  # noqa: E402

OUT = Path(__file__).resolve().parent


def main():
    require_reference()
    strict, orc = CpuTracer("ref_strict"), CpuTracer("oracle")
    z = np.load(OUT / "robot_scene.npz")
    mats = [dict(ambient_coeff=tuple(r[0:3]), diffuse=tuple(r[3:6]), specular=tuple(r[6:9]), emission=tuple(r[9:12]),
                 reflection=float(r[12]), roughness=float(r[13]), ns=float(r[14]), specular_threshold=float(r[15])) for r in z["materials"]]
    robot = dict(xyz9=z["xyz9"], uv6=z["uv6"], mat=z["mat"], materials=mats)
    table = common.raster_table(robot)
    background = 0xff000000 | (135 << 16) | (206 << 8) | 235
    out = {}
    for name in common.RASTER_PINNED:
        scene, kw, m, tex, cam = table[name]
        ref_img, rand_values = common.oracle_renderer(strict, scene, kw, m, tex, cam=cam).raster(srand_seed=common.RASTER_SRAND)
        seeds = common.ssao_reference_seeds(rand_values)
        o = common.oracle_renderer(orc, scene, kw, m, tex, cam=cam)
        got, counters = o.raster(ref_seeds9=seeds if kw.get("enable_ssao") else None)
        assert np.array_equal(got, ref_img), name
        out[name + "_reference"] = ref_img
        if kw.get("enable_ssao"):
            out[name + "_seeds9"] = seeds
            out[name + "_per_pixel"] = o.raster()[0]
        print(f"{name}: {ref_img.shape}, oracle bit-exact, {(ref_img != background).mean() * 100:.1f}% of the pixels covered, {counters}")
    np.savez_compressed(OUT / "golden_raster.npz", **out)
    print("golden_raster.npz", (OUT / "golden_raster.npz").stat().st_size, "bytes")


if __name__ == "__main__":
    main()
