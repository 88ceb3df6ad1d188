"""ESRI float grid I/O of the harness (the format of the reference's DEMs, soil maps and saved states)."""
from pathlib import Path

import numpy as np
import pytest

from criteria3d_b200.raster import EsriGrid, layer_to_grid, read_flt, write_flt
from criteria3d_b200.synth import Catchment


def test_flt_roundtrip(tmp_path):
    vals = np.arange(12, dtype=np.float32).reshape(3, 4)
    vals[1, 2] = -9999
    g = EsriGrid(vals, 641947.15, 5724524.79, 2.0, -9999.0)
    write_flt(tmp_path / "dem.flt", g)
    r = read_flt(tmp_path / "dem.flt")
    assert np.array_equal(r.values, vals) and r.cell == 2.0 and r.nodata == -9999.0
    assert r.valid.sum() == 11 and abs(r.xll - g.xll) < 1e-9


def test_layer_to_grid_places_values_by_cell_rank():
    valid = np.array([[True, False, True], [True, True, False]])
    cat = Catchment(2, 3, 2, valid=valid)
    layer = np.array([10.0, 11.0, 12.0, 13.0])
    like = EsriGrid(np.zeros((2, 3), np.float32), 0, 0, 10.0, -9999.0)
    g = layer_to_grid(layer, cat.cell_rank, like)
    assert np.array_equal(g.values, np.array([[10, -9999, 11], [12, 13, -9999]], np.float32))
    assert cat.n_surface == 4 and cat.rain_sink_source(3.6).shape == (4,)


# ---- slope / aspect / runoff boundary (SURVEY 8 f2): numpy restatement vs the reference's own gis code -------------
GOLDEN = Path(__file__).parent / "golden"
GIS_REF = Path(__file__).resolve().parent.parent / "oracle" / "_ref" / "libgis_ref.so"


def _ours(dem, cell):
    from criteria3d_b200.raster import boundary_runoff, boundary_slope_tan, slope_aspect
    slope, aspect = slope_aspect(dem, cell)
    return slope, aspect, boundary_runoff(dem, aspect), boundary_slope_tan(slope)


def test_slope_aspect_boundary_match_reference_golden():
    """bundled STH DEM (config 1): bit-identical float maps and boundary mask (golden from the reference's gis.cpp)"""
    with np.load(GOLDEN / "config1_sth_inputs.npz") as z:
        dem, cell = z["dem"], float(z["cell"])
    with np.load(GOLDEN / "gis_sth.npz") as g:
        slope, aspect, boundary, tan = _ours(dem, cell)
        valid = dem != np.float32(-9999)
        assert np.array_equal(slope, g["slope"]) and np.array_equal(aspect, g["aspect"])
        assert np.array_equal(boundary, g["boundary"]) and int(boundary.sum()) > 0
        assert np.array_equal(tan[valid], g["tan"][valid])


def _cases():
    rng = np.random.default_rng(11)
    ragged = (200 + rng.random((61, 47)) * 30).astype(np.float32)
    ragged[rng.random(ragged.shape) < 0.15] = -9999
    bowl = (np.hypot(*np.mgrid[-8:9, -10:11]) * 0.7 + 50).astype(np.float32)          # strict minimum in the middle
    bowl[0:3, 0:4] = -9999
    return {"ragged": (ragged, 10.0), "flat": (np.full((9, 9), 100, np.float32), 5.0), "bowl": (bowl, 2.0),
            "one row": ((100 + np.arange(12, dtype=np.float32))[None, :], 4.0), "one cell": (np.full((1, 1), 7, np.float32), 1.0),
            "all nodata": (np.full((4, 5), -9999, np.float32), 3.0)}


@pytest.mark.skipif(not GIS_REF.exists(), reason="oracle/_ref/libgis_ref.so not built (make -C oracle ref REF=<CRITERIA3D checkout>)")
@pytest.mark.parametrize("name", sorted(_cases()))
def test_slope_aspect_boundary_match_reference_library(name):
    import sys
    sys.path.insert(0, str(GOLDEN))
    from make_golden import gis_reference
    dem, cell = _cases()[name]
    ours, ref = _ours(dem, cell), gis_reference(dem, cell)
    valid = dem != np.float32(-9999)
    for a, b, what in zip(ours[:3], ref[:3], ("slope", "aspect", "boundary")):
        assert np.array_equal(a, b), what
    assert np.array_equal(ours[3][valid], ref[3][valid])


@pytest.mark.skipif(not (GIS_REF.exists() and Path("/root/reference/DATA/DEM/DEM_Ravone.flt").exists()), reason="reference data absent")
def test_slope_aspect_boundary_ravone_dem():
    """the 519 x 1208 Ravone DEM shipped with the reference (422 282 valid cells)"""
    import sys
    sys.path.insert(0, str(GOLDEN))
    from make_golden import gis_reference
    from criteria3d_b200.raster import read_flt
    g = read_flt("/root/reference/DATA/DEM/DEM_Ravone.flt")
    ours, ref = _ours(g.values, g.cell), gis_reference(g.values, g.cell)
    for a, b in zip(ours[:3], ref[:3]):
        assert np.array_equal(a, b)


# ---- ESRI grid I/O against the reference's own reader / writer (agrolib/gis/gisIO.cpp) -------------------------------
def _ref_read(noext, cap=4_000_000):
    import ctypes as C
    lib = C.CDLL(str(GIS_REF))
    r, c, cell, xll, yll, flag = C.c_int(), C.c_int(), C.c_double(), C.c_double(), C.c_double(), C.c_float()
    v = np.empty(cap, np.float32)
    rc = lib.gisref_read_flt(str(noext).encode(), C.byref(r), C.byref(c), C.byref(cell), C.byref(xll), C.byref(yll), C.byref(flag),
                             v.ctypes.data_as(C.POINTER(C.c_float)), C.c_long(cap))
    assert rc == 0
    return v[: r.value * c.value].reshape(r.value, c.value).copy(), (cell.value, xll.value, yll.value, flag.value)


@pytest.mark.skipif(not GIS_REF.exists(), reason="oracle/_ref/libgis_ref.so not built (make -C oracle ref REF=<CRITERIA3D checkout>)")
def test_flt_files_interchange_with_the_reference_reader_and_writer(tmp_path):
    import ctypes as C
    vals = np.arange(35, dtype=np.float32).reshape(5, 7) * 1.25
    vals[2, 3] = -9999
    # ours written -> the reference reads the same grid and header
    write_flt(tmp_path / "ours.flt", EsriGrid(vals, 641947.15, 5724524.79, 2.5, -9999.0))
    data, hdr = _ref_read(tmp_path / "ours")
    assert np.array_equal(data, vals) and hdr == (2.5, 641947.15, 5724524.79, -9999.0)
    # the reference writes -> ours reads; identical payload bytes.  (The reference's header writer prints coordinates with
    # ofstream's default 6 significant digits, gisIO.cpp:1476-1483; ours keeps them in full.)
    lib = C.CDLL(str(GIS_REF))
    rc = lib.gisref_write_flt(str(tmp_path / "theirs").encode(), 5, 7, C.c_double(2.5), C.c_double(641947.15), C.c_double(5724524.79),
                              C.c_float(-9999), vals.ctypes.data_as(C.POINTER(C.c_float)))
    assert rc == 0
    g = read_flt(tmp_path / "theirs.flt")
    assert np.array_equal(g.values, vals) and g.cell == 2.5 and g.nodata == -9999.0
    assert (tmp_path / "theirs.flt").read_bytes() == (tmp_path / "ours.flt").read_bytes()


@pytest.mark.skipif(not (GIS_REF.exists() and Path("/root/reference/DATA/PROJECT/STH/MAPS/DEM_STH.flt").exists()), reason="reference data absent")
def test_bundled_dem_reads_like_the_reference_reader():
    data, hdr = _ref_read("/root/reference/DATA/PROJECT/STH/MAPS/DEM_STH")
    g = read_flt("/root/reference/DATA/PROJECT/STH/MAPS/DEM_STH.flt")
    assert np.array_equal(data, g.values) and hdr == (g.cell, g.xll, g.yll, np.float32(g.nodata))
    with np.load(GOLDEN / "config1_sth_inputs.npz") as z:          # the committed inputs of config 1 are this file
        assert np.array_equal(z["dem"], g.values)
