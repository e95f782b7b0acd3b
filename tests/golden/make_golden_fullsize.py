"""Cuts tests/golden/golden_fullsize.npz: BASELINE.json's configs at their FULL sizes, from the UNMODIFIED reference
compiled in this container (oracle/_ref/libref_strict.so; libref.so = the reference's own FMA flags for the CRCs).

    python tests/golden/make_golden_fullsize.py        (needs the original sources: RTB200_REFERENCE, see make_golden.py; ~2 minutes)

Per frame: the CRC32 of the whole ARGB32 image (pins the oracle bit-exactly on the CPU side), every FULL_ROW_STEP-th
row (what the GPU frame is compared with, within the north-star tolerance), and the ray counts.
  cfg1_full  robot, 1280x720, 1 shadow ray per hit
  cfg2_full  + 2048^2 u8 diffuse / AO / normal maps, ssaa_factor 2  (rows of the RESOLVED 1280x720 frame)
  cfg3_full  1920x1080, 16-ray rough-reflection fan, max_recursion_depth 1, roughness map, 4096x2048 sky, rng_seed 7
  cfg5_band  1 M-triangle hair ball, 3840x2160, shadows: rows HAIR_BAND of the frame
"""
from __future__ import annotations

import sys
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle.bindings import CpuTracer  # noqa: E402
from tests.conftest import require_reference  # noqa: E402
from raytracercpp_b200 import scenes  # noqa: E402
from raytracercpp_b200.renderer import precompute_materials  # noqa: E402
from tests import common  # noqa: E402

OUT = Path(__file__).resolve().parent


def crc(img):
    return np.uint32(zlib.crc32(np.ascontiguousarray(img, np.uint32).tobytes()))


def main():
    require_reference()
    strict, fma = CpuTracer("ref_strict"), CpuTracer("ref")
    z = np.load(OUT / "robot_scene.npz")
    rows = z["materials"]
    mats = [dict(ambient_coeff=tuple(r[0:3]), diffuse=tuple(r[3:6]), specular=tuple(r[6:9]), emission=tuple(r[9:12]),
                 reflection=float(r[12]), roughness=float(r[13]), ns=float(r[14]), specular_threshold=float(r[15])) for r in rows]
    robot = dict(xyz9=z["xyz9"], uv6=z["uv6"], mat=z["mat"])
    out = {}
    for name, (kw, m, tex) in common.fullsize_table(mats).items():
        t0 = time.time()
        img = common.oracle_image(strict, robot, kw, m, tex)          # seeded pixel loop + the reference's own downscale
        img_fma = common.oracle_image(fma, robot, kw, m, tex)
        r = common.oracle_renderer(strict, robot, kw, m, tex)
        r.trace_rows(want_image=False)
        out[name + "_crc"], out[name + "_crc_fma"] = crc(img), crc(img_fma)
        out[name + "_rows"] = img[::common.FULL_ROW_STEP].copy()
        out[name + "_hits"] = np.int64(r.last_hit_count())
        print(f"{name}: {img.shape} crc {int(out[name + '_crc']):08x} (fma build {int(out[name + '_crc_fma']):08x}), "
              f"{(img == img_fma).mean() * 100:.3f}% pixels equal between the builds, hits {int(out[name + '_hits'])}, {time.time() - t0:.1f} s")
    # cfg5: a band of the 4K hair frame
    xyz9, uv6, mat = scenes.hair_ball(**common.HAIR_FULL)
    scene = dict(xyz9=xyz9, uv6=uv6, mat=mat)
    hmats = precompute_materials([scenes.DEFAULT_SPHERE_MATERIAL])
    r = common.oracle_renderer(strict, scene, common.HAIR_KW, hmats, {})
    b0, b1, bs = common.HAIR_BAND
    t0 = time.time()
    sup, _ = r.trace_rows(row_begin=b0, row_end=b1, row_step=bs)
    out["cfg5_band_rows"] = sup[b0:b1:bs].copy()
    out["cfg5_band_crc"] = crc(out["cfg5_band_rows"])
    out["cfg5_band_hits"] = np.int64(r.last_hit_count())
    print(f"cfg5_band: {len(xyz9)} triangles, rows {b0}:{b1}:{bs}, crc {int(out['cfg5_band_crc']):08x}, hits {int(out['cfg5_band_hits'])}, {time.time() - t0:.1f} s")
    np.savez_compressed(OUT / "golden_fullsize.npz", **out)
    print("golden_fullsize.npz", (OUT / "golden_fullsize.npz").stat().st_size, "bytes")


if __name__ == "__main__":
    main()
