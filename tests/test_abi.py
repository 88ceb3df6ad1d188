"""Every symbol declared in include/sf3d.h is exported by each built library (no compute calls:
runs without a GPU), and the product refuses to run without a CUDA device instead of falling back."""
import ctypes
import re
from pathlib import Path

import pytest

from criteria3d_b200 import PRODUCT_LIB
from oracle import ORACLE_LIB, REFERENCE_LIB
from criteria3d_b200.capi import ALL_SYMBOLS

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "sf3d.h").read_text()
DECLARED = sorted(set(re.findall(r"\b(sf3d_[a-z0-9_]+)\s*\(", HEADER)))


def test_header_and_binding_agree():
    assert DECLARED == sorted(ALL_SYMBOLS)
    assert len(DECLARED) >= 80


@pytest.mark.parametrize("lib", [PRODUCT_LIB, ORACLE_LIB, REFERENCE_LIB], ids=["product", "oracle", "reference"])
def test_library_exports_every_declared_symbol(lib):
    if not lib.exists():
        if lib == REFERENCE_LIB:
            pytest.skip("oracle/_ref not built (make -C oracle ref REF=<CRITERIA3D checkout>)")
        pytest.fail(f"{lib} missing: run __graft_entry__.build()")
    h = ctypes.CDLL(str(lib), mode=ctypes.RTLD_LOCAL)
    missing = [s for s in DECLARED if not hasattr(h, s)]
    assert not missing, missing


def test_cpp_dropin_symbols_exported():
    """The product also exports the reference's C++ API (namespace soilFluxes3D::v2), mangled."""
    import subprocess
    out = subprocess.run(["nm", "-DC", str(PRODUCT_LIB)], capture_output=True, text=True, check=True).stdout
    for name in ("initializeSF3D", "setNode", "setNodeLink", "computeStep", "computePeriod", "getNodeWaterContent",
                 "getTotalBoundaryWaterFlow", "setNodeWaterSinkSource", "getNodeHeatMaxFlux", "setCulvert"):
        assert f"soilFluxes3D::v2::{name}(" in out, name


def test_product_has_no_cpu_fallback():
    """Without a CUDA device sf3d_initialize must fail (MemoryError), not compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from criteria3d_b200 import SoilFluxes3D
    sf = SoilFluxes3D(PRODUCT_LIB)
    assert sf.backend == "b200"
    assert sf.initializeSF3D(10, 2, 8, True, False, False, 0) != 0
    assert sf.computeStep(10.0) == -2222.0          # not initialised -> MemoryError sentinel


def test_product_does_not_link_or_reference_the_oracle():
    import subprocess
    out = subprocess.run(["ldd", str(PRODUCT_LIB)], capture_output=True, text=True).stdout
    assert "sf3d_oracle" not in out and "sf3d_ref" not in out
    # no file of the product package names the oracle libraries, imports the oracle package or includes oracle
    # files: the checkers' paths live in oracle/__init__.py (test infrastructure)
    tokens = ("libsf3d_oracle", "libsf3d_ref", "ORACLE_LIB", "REFERENCE_LIB", "oracle/sf3d", "oracle/ref_capi", "grid_builder_scalar",
              "from oracle", "import oracle")
    for src in (ROOT / "criteria3d_b200").rglob("*"):
        if src.suffix in (".cu", ".cpp", ".h", ".py"):
            text = src.read_text()
            assert not any(t in text for t in tokens), src


def test_raster_preparation_symbol_exported():
    """include/sf3d_gis.h (SURVEY 8 f2): declared symbols are exported by the product (no compute call here)"""
    hdr = (ROOT / "include" / "sf3d_gis.h").read_text()
    declared = sorted(set(re.findall(r"\b(sf3d_gis_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == ["sf3d_gis_slope_aspect_boundary"]
    h = ctypes.CDLL(str(PRODUCT_LIB), mode=ctypes.RTLD_LOCAL)
    assert all(hasattr(h, s) for s in declared)
