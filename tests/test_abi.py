"""The C-ABI library: builds for sm_100a, loads, exports every symbol include/rtb200.h declares, and refuses to run
without a CUDA device (no CPU fallback).  No compute calls here."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

from raytracercpp_b200 import api, build
from tests.conftest import REFERENCE, cuda_available

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return api.load_library()


def declared_symbols():
    text = (ROOT / "include" / "rtb200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rt_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    syms = declared_symbols()
    assert len(syms) >= 25
    raw = ctypes.CDLL(str(api.LIB_PATH))
    for s in syms:
        assert hasattr(raw, s), f"{s} declared in include/rtb200.h but not exported"
    assert set(api.ABI) == set(syms)


def test_struct_sizes(lib):
    assert ctypes.sizeof(api.RtMaterial) == 64
    assert ctypes.sizeof(api.RtSettings) == 31 * 4


def test_defaults_mirror_render_settings(lib):
    s = api.default_settings(lib)                      # rendererSettings.h:29-102
    assert (s.image_width, s.image_height, s.ssaa_factor, s.max_recursion_depth) == (1024, 1024, 2, 5)
    assert (s.enable_bvh, s.bvh_max_depth, s.bvh_leaf_object_count, s.rough_reflections_sample_count) == (1, 12, 40, 3)
    assert abs(s.displacement_mapping_strength - 0.02) < 1e-9 and s.parallax_mapping_steps == 32      # rendererSettings.h:94-95
    assert (s.ssao_sample_count, s.ssao_radius, s.ssao_amount) == (64, 0.5, 1.0) and not s.enable_ssao    # rendererSettings.h:66-73
    assert s.enable_ambient and s.enable_diffuse and s.enable_specular and s.enable_emissive
    assert s.enable_clipping and not s.hybrid_rasterization_tracing                                     # rendererSettings.h:40,46
    assert not (s.enable_ssaa or s.compute_shadows or s.enable_skysphere or s.enable_ao_mapping)


@pytest.mark.skipif(cuda_available(), reason="this container-side check needs the absence of a GPU")
def test_no_cpu_fallback(lib):
    with pytest.raises(api.RtError) as e:
        api.Context(0, lib)
    assert e.value.code == api.RT_ERR_CUDA
    assert "no CPU path" in e.value.message


def test_host_helpers_match_oracle(lib, oracle, golden_images):
    out = np.zeros(16, np.float32)
    lib.rt_perspective_inverse(80.0, 16.0 / 9.0, 0.1, 1000.0, out.ctypes.data_as(api.FP))
    assert np.array_equal(out.reshape(4, 4), golden_images["proj_inv_80_16x9"])
    m = np.ascontiguousarray(golden_images["inv_in"].reshape(16))
    lib.rt_invert_transform(m.ctypes.data_as(api.FP), out.ctypes.data_as(api.FP))
    assert np.array_equal(out.reshape(4, 4), golden_images["inv_out"])
    assert lib.rt_pixel_seed(0, 0) == 1 and lib.rt_pixel_seed(12345, 7) % 2 == 1


def test_tile_ownership_is_a_partition(lib):
    s = api.default_settings(lib, image_width=1000, image_height=600)
    for tile in (32, 64, 100):
        total = (1000 + tile - 1) // tile * ((600 + tile - 1) // tile)
        for mod in (1, 2, 3, 8):
            counts = [lib.rt_tile_count(ctypes.byref(s), tile, mod, r) for r in range(mod)]
            assert sum(counts) == total and max(counts) - min(counts) <= 2
    assert lib.rt_tile_count(ctypes.byref(s), 64, 2, 2) == api.RT_ERR_INVALID


def test_adapter_compiles_against_the_reference_headers(tmp_path):
    """include/rtb200_renderer.hpp with the reference's REAL Triangle / Materials / Image / Transform / Point / Vector
    (headers included from the original sources where they lie; Qt's QImage from the oracle's shim): every templated
    member is instantiated with them.  CPU-only object file; needs the original sources (RTB200_REFERENCE)."""
    import subprocess
    ref = REFERENCE
    if ref is None or not (ref / "projets" / "triangle.h").exists():
        pytest.skip("the original sources are not here (RTB200_REFERENCE)")
    obj = tmp_path / "adapter_reference_types.o"
    inc = [ROOT / "include", ROOT / "oracle" / "qt_shim", ref / "src", ref / "projets", ref / "projets" / "utils", ref / "projets" / "renderer",
           ref / "projets" / "scene"]
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-c", "-o", str(obj), str(ROOT / "tests" / "adapter_reference_types.cpp")] + [f"-I{p}" for p in inc]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    syms = subprocess.run(["nm", "-C", str(obj)], capture_output=True, text=True, check=True).stdout
    for member in ("set_triangles<Triangle>", "set_materials<Materials>", "set_ao_map<Image>", "set_skybox<Image>", "set_camera_transform<Transform>",
                   "set_object_transform<Transform>", "set_light_position<Point>", "add_plane<Point, Vector>", "copy_to<QImage>"):
        assert f"rtb200::Renderer::{member}" in syms, member
