"""Shared fixtures.

Markers: `gpu` = needs a CUDA device and goes through librtb200.so (the parity tests proper);
everything else runs on the CPU: the oracle against the golden vectors cut from the compiled reference, the host
logic, the ABI surface of the CUDA library, and the kernels' per-ray source compiled for the host (tests/hostsim).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

GOLDEN = ROOT / "tests" / "golden"
# The original RayTracerCPP sources (its tp2 directory) are not part of this repository.  The live comparisons with them
# run where RTB200_REFERENCE names that directory (`make -C oracle ref` compiles it into oracle/_ref) and skip elsewhere;
# the committed goldens under tests/golden carry what they were compared against.
REFERENCE = Path(os.environ["RTB200_REFERENCE"]) if os.environ.get("RTB200_REFERENCE") else None


def require_reference() -> Path:
    """For the golden generators (tests/golden/make_golden*.py): the original's tp2 directory, or a clear stop."""
    if REFERENCE is None or not REFERENCE.is_dir():
        raise SystemExit("the original sources are needed: export RTB200_REFERENCE=<RayTracerCPP>/tp2, then make -C oracle ref")
    return REFERENCE


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _make(directory: Path, target: str):
    subprocess.run(["make", "-s", "-C", str(directory), target], check=True)


def cuda_available() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def oracle():
    from oracle import bindings
    if not bindings.available("oracle"):
        _make(ROOT / "oracle", "liboracle.so")
    return bindings.CpuTracer("oracle")


@pytest.fixture(scope="session")
def ref_strict():
    from oracle import bindings
    if not bindings.available("ref_strict"):
        pytest.skip("oracle/_ref/libref_strict.so not built (needs the original sources, RTB200_REFERENCE)")
    return bindings.CpuTracer("ref_strict")


@pytest.fixture(scope="session")
def ref_fma():
    from oracle import bindings
    if not bindings.available("ref"):
        pytest.skip("oracle/_ref/libref.so not built (needs the original sources, RTB200_REFERENCE)")
    return bindings.CpuTracer("ref")


@pytest.fixture(scope="session")
def hostsim_lib():
    """The kernels' per-ray source compiled for the CPU behind the same C ABI (test infrastructure only)."""
    from raytracercpp_b200 import api
    _make(ROOT / "tests" / "hostsim", "librtb200_hostsim.so")
    return api.bind(ctypes.CDLL(str(ROOT / "tests" / "hostsim" / "librtb200_hostsim.so")))


@pytest.fixture(scope="session")
def cuda_lib():
    from raytracercpp_b200 import api
    if not cuda_available():
        pytest.skip("no CUDA device")
    return api.load_library()


@pytest.fixture(scope="session")
def robot():
    z = np.load(GOLDEN / "robot_scene.npz")
    rows = z["materials"]
    mats = [dict(ambient_coeff=tuple(r[0:3]), diffuse=tuple(r[3:6]), specular=tuple(r[6:9]), emission=tuple(r[9:12]),
                 reflection=float(r[12]), roughness=float(r[13]), ns=float(r[14]), specular_threshold=float(r[15])) for r in rows]
    return dict(xyz9=z["xyz9"], uv6=z["uv6"], mat=z["mat"], materials=mats)


@pytest.fixture(scope="session")
def golden_ssao():
    return dict(np.load(GOLDEN / "golden_ssao.npz"))


@pytest.fixture(scope="session")
def golden_raster():
    return dict(np.load(GOLDEN / "golden_raster.npz"))


@pytest.fixture(scope="session")
def golden_rays():
    return dict(np.load(GOLDEN / "golden_rays.npz"))


@pytest.fixture(scope="session")
def golden_images():
    return dict(np.load(GOLDEN / "golden_images.npz"))


@pytest.fixture(scope="session")
def golden_fullsize():
    return dict(np.load(GOLDEN / "golden_fullsize.npz"))
