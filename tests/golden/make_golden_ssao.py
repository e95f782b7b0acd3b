"""Cuts tests/golden/golden_ssao.npz: SSAO frames (renderer.cpp:1229-1434) from the UNMODIFIED reference compiled in this
container (oracle/_ref/libref_strict.so), its SSAO pass run on one thread after srand(SRAND_SEED) -- the only reproducible
way to run it: its generators are seeded from std::rand() and the OpenMP thread number.

    python tests/golden/make_golden_ssao.py        (needs the original sources: RTB200_REFERENCE, see make_golden.py)

Per set-up of tests/common.py::ssao_table: the reference's frame, the nine generator seeds that run used (lanes 0..7 of the
8-lane generator, the scalar generator), and the oracle's frame with the per-pixel stream the CUDA path shares.
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
SRAND_SEED = 20261019


def main():
    require_reference()
    strict, orc = CpuTracer("ref_strict"), CpuTracer("oracle")
    z = np.load(OUT / "robot_scene.npz")
    mats = [dict(ambient_coeff=tuple(r[0:3]), diffuse=tuple(r[3:6]), specular=tuple(r[6:9]), emission=tuple(r[9:12]),
                 reflection=float(r[12]), roughness=float(r[13]), ns=float(r[14]), specular_threshold=float(r[15])) for r in z["materials"]]
    robot = dict(xyz9=z["xyz9"], uv6=z["uv6"], mat=z["mat"])
    out = {}
    for name, (kw, m, tex) in common.ssao_table(mats).items():
        ref_img, rand_values = common.oracle_renderer(strict, robot, kw, m, tex).render_ssao(srand_seed=SRAND_SEED)
        seeds = common.ssao_reference_seeds(rand_values)
        o = common.oracle_renderer(orc, robot, kw, m, tex)
        got, _ = o.render_ssao(ref_seeds9=seeds)
        per_pixel, _ = o.render_ssao()
        assert np.array_equal(got, ref_img), name
        out[name + "_reference"], out[name + "_seeds9"], out[name + "_per_pixel"] = ref_img, seeds, per_pixel
        print(f"{name}: {ref_img.shape}, oracle (reference order) bit-exact, per-pixel stream differs on {(per_pixel != ref_img).mean() * 100:.1f}% of the pixels")
    np.savez_compressed(OUT / "golden_ssao.npz", **out)
    print("golden_ssao.npz", (OUT / "golden_ssao.npz").stat().st_size, "bytes")


if __name__ == "__main__":
    main()
