"""Cuts tests/golden/golden_obj.npz: what the UNMODIFIED reference's loader (read_meshio_data + MeshIOUtils::create_triangles,
tp2/src/mesh_io.cpp:426-591, tp2/projets/utils/meshIOUtils.cpp:4-33; compiled into oracle/_ref/libref_strict.so) makes of the
fixture files under tests/golden/obj/ -- triangles, texture coordinates, material indices, material table -- for the
parity test of csrc/scene_io.cpp (tests/test_scene_io.py).

    python tests/golden/make_golden_obj.py        (needs the original sources: RTB200_REFERENCE, see make_golden.py)
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.bindings import CpuTracer  # noqa: E402
from tests.conftest import require_reference  # noqa: E402

OUT = Path(__file__).resolve().parent
TRANSFORM = np.float32([[0.5, 0, 0, 0.25], [0, 2.0, 0, -2.0], [0, 0, 1.0, -4.0], [0, 0, 0, 1]])


def rows(mats):
    return np.float32([list(m["ambient_coeff"]) + list(m["diffuse"]) + list(m["specular"]) + list(m["emission"]) +
                       [m["reflection"], m["roughness"], m["ns"]] for m in mats]).reshape(len(mats), 15)


def main():
    require_reference()
    strict = CpuTracer("ref_strict")
    out = {"transform": TRANSFORM}
    for name, tr in (("fixture_uv", TRANSFORM), ("fixture_plain", None)):
        xyz9, uv6, mat, mats = strict.load_obj(str(OUT / "obj" / (name + ".obj")), tr)
        out[name + "_xyz9"], out[name + "_uv6"], out[name + "_mat"], out[name + "_materials"] = xyz9, uv6, mat, rows(mats)
        print(name, xyz9.shape, "materials", len(mats), "indices", sorted(set(mat.tolist())))
    np.savez_compressed(OUT / "golden_obj.npz", **out)


if __name__ == "__main__":
    main()
