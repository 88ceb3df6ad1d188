"""Seeded scenarios shared by the CPU (oracle vs reference / golden) and GPU (product vs oracle)
parity tests.  Each scenario drives ONE implementation of the C ABI and returns a dict of
arrays/scalars to compare.  Edge cases follow what the reference's code paths distinguish:
retention model and mean type, evaporation clamp, prescribed-potential / urban / road boundaries,
saturated columns, ragged (NODATA) rasters, scalar-API graphs, empty forcing."""
from __future__ import annotations

import numpy as np

from criteria3d_b200 import BoundaryType, Field, LinkType, MeanType, WRCModel
from criteria3d_b200.synth import Catchment, run_hours, set_heat_forcing, setup, setup_heat, _ok

FIELDS = (Field.TOTAL_POTENTIAL, Field.WATER_CONTENT, Field.DEGREE_OF_SATURATION, Field.WATER_CONDUCTIVITY,
          Field.BOUNDARY_WATER_FLOW, Field.MAX_FLOW_UP, Field.MAX_FLOW_DOWN, Field.SUM_LATERAL_FLOW)


def snapshot(sf, n_nodes, dts, n_surface=None):
    out = {f.name: sf.get_field(f, 0, n_nodes) for f in FIELDS}
    out["n_surface"] = np.int64(sf.node_meta(0, n_nodes)[0].sum())
    out["dts"] = np.asarray(dts, dtype=np.float64)
    out["total_water"] = np.float64(sf.getTotalWaterContent())
    out["boundary_totals"] = np.array([sf.getTotalBoundaryWaterFlow(int(b)) for b in
                                       (BoundaryType.Runoff, BoundaryType.FreeDrainage,
                                        BoundaryType.FreeLateralDrainage, BoundaryType.PrescribedTotalWaterPotential)])
    c = sf.counters()
    out["counters"] = np.array([c["approximations"], c["sweeps"]], dtype=np.float64)
    out["mbe_mbr"] = np.array([c["last_mbe"], c["last_mbr"], c["delta_t_curr"], c["last_courant"]])
    out["storage"] = np.float64(sf.getWaterStorage())
    return out


def heat_snapshot(sf, cat, out):
    """temperatures and heat-boundary diagnostics of a coupled run (soil nodes only)"""
    ns, n = cat.n_surface, cat.n_nodes
    out["TEMPERATURE"] = sf.get_field(Field.TEMPERATURE, ns, n - ns)
    probe = range(ns, 2 * ns, max(1, ns // 7))
    out["heat_boundary"] = np.array([[sf.getNodeBoundarySensibleFlux(i), sf.getNodeBoundaryLatentFlux(i),
                                      sf.getNodeBoundaryRadiativeFlux(i), sf.getNodeBoundaryAerodynamicConductance(i),
                                      sf.getNodeBoundarySoilConductance(i), sf.getNodeHeatConductivity(i),
                                      sf.getNodeHeatStorage(i, -1.0), sf.getNodeVapor(i)] for i in probe])
    out["heat_flux_down"] = np.array([sf.getNodeHeatMaxFlux(i, 2, 0) for i in range(2 * ns, 3 * ns)])
    c = sf.counters()
    out["heat_counters"] = np.array([c["heat_steps"], c["heat_sweeps"]], dtype=np.float64)
    out["heat_cap_hits"] = np.float64(c["heat_cap_hits"])      # heat solves that ended at the sweep cap (Q6)
    out["heat_mbr_mbe"] = np.array([sf.getHeatMBR(), sf.getHeatMBE()])
    return out


def heat_coupled(sf, threads=1, latent=True):
    """C3-like: coupled heat (diffusive + latent; see synth.setup_heat for why advection is off),
    a dry hour with sun then an hour of rain, atmospheric forcing changing per hour"""
    cat = Catchment(10, 8, 4, heat=True)
    setup(sf, cat, threads=threads)
    if not latent:
        _ok(sf.initializeHeatFlag(1, False, False), "initializeHeatFlag")
        _ok(sf.initializeBalance(), "balance")
    dts = []
    for h, mm in ((10, 0.0), (11, 10.0)):
        set_heat_forcing(sf, cat, h)
        dts += run_hours(sf, cat, [mm], max_steps=12)
    return heat_snapshot(sf, cat, snapshot(sf, cat.n_nodes, dts))


def heat_coupled_medium(sf, threads=1):
    """coupled heat (diffusive + latent) past toy size: 32 x 32 x (1+10) = 11 264 nodes, a dry sunny hour and the
    first 12 accepted steps of a 20 mm/h rain hour (about 400 heat sub-steps, 2 500 heat sweeps; ~45 s for the
    reference on one thread, which is why it is a GPU-suite case without a committed golden vector)"""
    cat = Catchment(32, 32, 10, heat=True)
    setup(sf, cat, threads=threads)
    dts = []
    for h, mm, budget in ((10, 0.0, 8), (11, 20.0, 12)):
        set_heat_forcing(sf, cat, h)
        dts += run_hours(sf, cat, [mm], max_steps=budget)
    return heat_snapshot(sf, cat, snapshot(sf, cat.n_nodes, dts))


def heat_diffusive_only(sf, threads=1):
    return heat_coupled(sf, threads=threads, latent=False)


def heat_advective_column(sf, threads=1, shape=(1, 1, 6), save_all=False, phases=((0.0, 10.0, 15), (1.0, 5.0, 12))):
    """SURVEY 3.4 / Appendix B Q1: a 6-layer column with a HeatSurface boundary on the first soil layer, a
    FreeDrainage + fixed-temperature bottom and initializeHeatFlag(.., advection = true, latent = true), so
    that computeAdvectiveFlux (heat.cpp:606-621, call site :442) and the advective boundary terms
    (heat.cpp:273-287 rain / evaporation, :302-309 drainage) are executed.  The reference's advective term is
    not conservative (Q1: the soil side of the infiltration link reports a normalised flux two orders of
    magnitude too large) and reaches NaN inside ONE default-length water step; bounded to short steps it stays
    finite and that trajectory is what is pinned: phases = (rain mm/h, max step s, computeStep calls): a dry
    phase (evaporation branch; top node 288.15 -> ~287 K) and a 1 mm/h rain phase (rain branch; the top node
    heats to ~330 K: unphysical, and exactly what the reference computes)."""
    cat = Catchment(*shape, heat=True)
    mode = 2 if save_all else 1
    setup(sf, cat, threads=threads, heat_flux_mode=mode)
    setup_heat(sf, cat, hour=10, advection=True, latent=True, mode=mode)
    _ok(sf.initializeBalance(), "balance")
    sink = np.zeros(cat.n_nodes)
    dts = []
    for mm, max_dt, steps in phases:
        sink[: cat.n_surface] = cat.rain_sink_source(mm)
        _ok(sf.set_field(Field.WATER_SINK_SOURCE, 0, sink), "sink")
        dts += [sf.computeStep(max_dt) for _ in range(steps)]
    out = heat_snapshot(sf, cat, snapshot(sf, cat.n_nodes, dts))
    ns = cat.n_surface
    out["heat_advective_boundary"] = np.array([sf.getNodeBoundaryAdvectiveFlux(i) for i in
                                               list(range(ns, 2 * ns)) + list(range(cat.n_nodes - ns, cat.n_nodes))])
    if save_all:
        # per-type link fluxes (fluxTypes_t, types.h:199): diffusive, latent isothermal / thermal, advective,
        # and the four water flux snapshots, Down direction, second soil layer
        out["heat_flux_types"] = np.array([[sf.getNodeHeatMaxFlux(i, 2, t) for t in range(9)] for i in range(2 * ns, 3 * ns)])
    assert np.all(np.isfinite(out["TEMPERATURE"])), "advective trajectory left the finite range"
    return out


def heat_advective_slope(sf, threads=1):
    """the same with lateral links (4 x 3 cells on a slope) and every flux type saved (HFsaveMode All)"""
    return heat_advective_column(sf, threads=threads, shape=(4, 3, 6), save_all=True)


def storm(sf, shape=(24, 20, 5), hours=(20.0, 40.0), threads=1, max_steps=60, **cat_kw):
    cat = Catchment(*shape, **cat_kw)
    setup(sf, cat, threads=threads)
    dts = run_hours(sf, cat, list(hours), max_steps=max_steps)
    return snapshot(sf, cat.n_nodes, dts)


def van_genuchten_geometric(sf, threads=1):
    """plain VG retention, geometric mean, horizontal/vertical ratio 5, looser numerics"""
    cat = Catchment(20, 16, 4)
    setup(sf, cat, threads=threads, numerics=(1.0, 1800.0, 100, 8, 9, 2))
    _ok(sf.setHydraulicProperties(int(WRCModel.VanGenuchten), int(MeanType.Geometric), 5.0), "hyd")
    _ok(sf.set_field(Field.MATRIC_POTENTIAL, 0, cat.initial_matric_potential()), "psi")   # Se/K under the new model
    _ok(sf.initializeBalance(), "balance")
    dts = run_hours(sf, cat, [30.0], max_steps=40)
    return snapshot(sf, cat.n_nodes, dts)


def evaporation_after_rain(sf, threads=1):
    """arithmetic mean; one wet hour, then a surface sink larger than the ponded water
    (evaporation clamp, water.cpp:645-652)"""
    cat = Catchment(18, 18, 4)
    setup(sf, cat, threads=threads)
    _ok(sf.setHydraulicProperties(int(WRCModel.ModifiedVanGenuchten), int(MeanType.Arithmetic), 10.0), "hyd")
    dts = run_hours(sf, cat, [15.0], max_steps=40)
    sink = np.zeros(cat.n_nodes)
    sink[: cat.n_surface] = -cat.rain_sink_source(3.0)
    _ok(sf.set_field(Field.WATER_SINK_SOURCE, 0, sink), "sink")
    t = 0.0
    while t < 1800.0 and len(dts) < 80:
        dt = sf.computeStep(1800.0 - t)
        dts.append(dt)
        t += dt
    return snapshot(sf, cat.n_nodes, dts)


def prescribed_and_urban(sf, threads=1):
    """bottom layer with a prescribed total potential (water table 0.5 m below the bottom nodes on
    the left half), Urban / Road cells on layer 1, no free bottom drainage"""
    cat = Catchment(16, 20, 4)
    bl1 = np.zeros((cat.rows, cat.cols), np.uint8)
    bl1[4:8, 3:9] = int(BoundaryType.Urban)
    bl1[10:13, 10:16] = int(BoundaryType.Road)
    cat.outlet[:] = 0
    cat.outlet[cat.rows - 1, :] = 1

    def grid_desc():
        d = Catchment.grid_desc(cat)
        d.boundary_l1 = bl1.ctypes.data_as(type(d.boundary_l1))
        d.free_bottom_drainage = 0
        return d
    cat.grid_desc = grid_desc
    setup(sf, cat, threads=threads)
    last = (cat.layers - 1) * cat.n_surface
    area = cat.cell * cat.cell
    H0 = sf.get_field(Field.TOTAL_POTENTIAL, 0, cat.n_nodes)
    for r in range(cat.rows):
        for c in range(cat.cols // 2):
            i = last + r * cat.cols + c
            _ok(sf.setNodeBoundary(i, int(BoundaryType.PrescribedTotalWaterPotential), 0.0, area), "bc")
            z = H0[i] - cat.initial_psi
            _ok(sf.setNodePrescribedTotalPotential(i, z - 0.5), "presc")
    assert sf.setNodePrescribedTotalPotential(0, 1.0) == 4          # BoundaryError on a non-prescribed node
    _ok(sf.initializeBalance(), "balance")
    dts = run_hours(sf, cat, [25.0], max_steps=40)
    return snapshot(sf, cat.n_nodes, dts)


def dry_no_forcing(sf, threads=1):
    """empty forcing: no rain, no sinks; redistribution and free drainage only, the time step grows to its
    maximum (doubling rule, water.cpp:197-200) and whole-hour steps are accepted"""
    cat = Catchment(12, 10, 4)
    setup(sf, cat, threads=threads)
    dts = run_hours(sf, cat, [0.0, 0.0, 0.0])
    return snapshot(sf, cat.n_nodes, dts)


def culvert_outlet(sf, threads=1):
    """Culvert boundary on part of the outlet row.  Unreachable in the reference (setCulvert writes through
    a pointer array that is never allocated, soilFluxes3D.cpp:146,586: SURVEY Q5), so this case pins the
    product against the C restatement of water.cpp:749-795 (mean-head form of v1) only."""
    cat = Catchment(14, 12, 3)
    setup(sf, cat, threads=threads)
    last_row = (cat.rows - 1) * cat.cols
    for c in range(3, 9):
        _ok(sf.setCulvert(last_row + c, 0.015, 0.02, 0.8, 0.5), "setCulvert")
    assert sf.setCulvert(cat.n_surface + 1, 0.015, 0.02, 0.8, 0.5) == 1          # soil node -> IndexError
    _ok(sf.initializeBalance(), "balance")
    dts = run_hours(sf, cat, [60.0], max_steps=60)
    out = snapshot(sf, cat.n_nodes, dts)
    out["culvert_total"] = np.float64(sf.getTotalBoundaryWaterFlow(int(BoundaryType.Culvert)))
    return out


def saturated_bottom(sf, threads=1):
    """C4-like: lower third of the layers start saturated (psi = +0.1 m)"""
    return storm(sf, shape=(20, 20, 9), hours=(10.0,), threads=threads, saturated_bottom=True)


def twenty_layers_saturated_mix(sf, threads=1):
    """C4 / C5 layering: 20 soil layers (thickness 0.02 .. 0.10 m, depth ~1.7 m: three horizons), the lower third
    saturated at the start, free drainage at the bottom, one storm hour"""
    return storm(sf, shape=(24, 24, 20), hours=(40.0,), threads=threads, max_steps=40, saturated_bottom=True)


def ragged_raster(sf, threads=1):
    """NODATA holes and a ragged edge: nodes with fewer than 8 lateral links"""
    valid = np.ones((22, 18), bool)
    valid[0:3, 0:5] = False
    valid[9:12, 7:10] = False
    valid[:, -1] = np.arange(22) % 3 != 0
    cat = Catchment(22, 18, 4, valid=valid)
    setup(sf, cat, threads=threads)
    dts = run_hours(sf, cat, [30.0], max_steps=40)
    return snapshot(sf, cat.n_nodes, dts)


def raster_forcing_and_maps(sf, threads=1):
    """the caller's side of the step through rasters (SURVEY 8 f3/f4): hourly precipitation map ->
    sink/source (assignPrecipitation + setSinkSource), then an evapotranspiration hour with per-layer
    sink maps (assignETreal), then output maps of four layers (computeCriteria3DMap)"""
    valid = np.ones((20, 17), bool)
    valid[0:2, 0:4] = False
    valid[8:10, 6:9] = False
    cat = Catchment(20, 17, 4, valid=valid)
    setup(sf, cat, threads=threads)
    dts = []

    def hour(seconds, budget):
        t = 0.0
        while t < seconds and len(dts) < budget:
            dt = sf.computeStep(seconds - t)
            dts.append(dt)
            t += dt

    _ok(sf.set_forcing_rasters(precipitation=cat.rain_raster(25.0)), "forcing rasters (rain)")
    hour(3600.0, 40)
    r, c = np.mgrid[0:cat.rows, 0:cat.cols]
    et = np.zeros((3, cat.rows, cat.cols), np.float32)
    et[0] = 0.6 + 0.2 * np.cos(r / 3.0)                 # surface evaporation [mm h-1]
    et[1] = 0.25 + 0.1 * np.sin(c / 2.0)                # first soil layer
    et[2] = np.where((r + c) % 3 == 0, 0.0, 0.1)        # second soil layer, zeros are skipped
    et[1, 5, 5] = -9999.0                               # a NODATA cell of the map is skipped
    _ok(sf.set_forcing_rasters(precipitation=np.zeros((cat.rows, cat.cols), np.float32), layer_sink=et), "forcing rasters (ET)")
    hour(1800.0, 70)
    out = snapshot(sf, cat.n_nodes, dts)
    shape = (cat.rows, cat.cols)
    out["rasters"] = np.stack([sf.get_layer_raster(Field.WATER_CONTENT, 0, shape), sf.get_layer_raster(Field.WATER_CONTENT, 2, shape),
                               sf.get_layer_raster(Field.DEGREE_OF_SATURATION, 1, shape), sf.get_layer_raster(Field.TOTAL_POTENTIAL, 4, shape),
                               sf.get_layer_raster(Field.MATRIC_POTENTIAL, 3, shape),
                               *sf.get_layer_rasters(Field.MATRIC_POTENTIAL, 0, cat.layers, shape)])      # saveModelsState
    return out


def config1_bundled_catchment(sf, threads=1, hours=8, max_steps=100):
    """BASELINE config 1: the bundled STH sample catchment (DATA/PROJECT/STH/MAPS/DEM_STH.flt, 34 x 139
    cells of 2 m, 1244 NODATA cells; soil map ids 1-3), water only, 2 mm/h rain.  The full 24 h run is
    17 841 accepted steps (dt is Courant-limited to ~5 s on 2 m cells; 15 min on one CPU thread), so the
    parity case is bounded to the first 100 accepted steps (about 5 simulated hours); bench-style full runs are left to the harness.
    The rasters are committed as tests/golden/config1_sth_inputs.npz (made by make_golden.py with
    criteria3d_b200/raster.py from the reference's DATA directory)."""
    from pathlib import Path
    with np.load(Path(__file__).parent / "golden" / "config1_sth_inputs.npz") as z:
        dem, soil, cell = z["dem"], z["soil"], float(z["cell"])
    valid = dem != np.float32(-9999)
    cat = Catchment(dem.shape[0], dem.shape[1], 5, cell=cell, valid=valid, dem_override=np.where(valid, dem, 0).astype(np.float32),
                    soil_override=np.where(valid, soil, 1).astype(np.uint16))
    setup(sf, cat, threads=threads)
    dts = run_hours(sf, cat, [2.0] * hours, max_steps=max_steps)
    return snapshot(sf, cat.n_nodes, dts)


def scalar_api_column(sf, threads=1):
    """A 3-column x 5-node graph built ONLY with the scalar API (CRITERIA-1D style), checking
    return codes on the way; then two hours of infiltration."""
    ncol, nlay = 3, 5
    ns, n = ncol, ncol * nlay
    sf.reset_solver()
    _ok(sf.initializeSF3D(n, ns, 8, True, False, False, 0), "init")
    _ok(sf.setSurfaceProperties(0, 0.05), "surf")
    _ok(sf.setSoilProperties(0, 0, 3.6, 1.56, 1 - 1 / 1.56, 0.02, 0.078, 0.43, 2.9e-6, 0.5, 0.02, 0.2), "soil")
    assert sf.setSoilProperties(0, 0, 3.6, 1.56, 1 - 1 / 1.56, 0.02, 0.078, 0.43, 2.9e-6, 0.5, 0.02, 0.2) == 6   # duplicate
    assert sf.setSoilProperties(1, 0, -1.0, 1.56, 0.3, 0.02, 0.078, 0.43, 2.9e-6, 0.5, 0.02, 0.2) == 6           # alpha <= 0
    thick = [0.0, 0.05, 0.10, 0.15, 0.20]
    depth = [0.0, 0.025, 0.10, 0.225, 0.40]
    area = 1.0
    for lay in range(nlay):
        for c in range(ncol):
            i = lay * ncol + c
            x, y, z = 1.0 * c, 0.0, 10.0 + 0.05 * c - depth[lay]
            if lay == 0:
                bt = int(BoundaryType.Runoff) if c == 0 else 0
                _ok(sf.setNode(i, x, y, z, area, True, bt, 0.05, 1.0), "setNode")
            elif lay == nlay - 1:
                _ok(sf.setNode(i, x, y, z, area * thick[lay], False, int(BoundaryType.FreeDrainage), 0.0, area), "setNode")
            else:
                _ok(sf.setNode(i, x, y, z, area * thick[lay], False, 0, 0.0, 0.0), "setNode")
    assert sf.setNode(n, 0, 0, 0, 1, True, 0, 0, 0) == 1                     # IndexError
    for lay in range(nlay):
        for c in range(ncol):
            i = lay * ncol + c
            if lay > 0:
                _ok(sf.setNodeLink(i, i - ncol, int(LinkType.Up), area), "up")
            if lay < nlay - 1:
                _ok(sf.setNodeLink(i, i + ncol, int(LinkType.Down), area), "down")
            for dc in (-1, 1):
                if 0 <= c + dc < ncol:
                    la = 0.5 if lay == 0 else 0.5 * thick[lay]
                    _ok(sf.setNodeLink(i, i + dc, int(LinkType.Lateral), la), "lat")
            if lay == 0:
                _ok(sf.setNodeSurface(i, 0), "surface")
                _ok(sf.setNodePond(i, 0.003), "pond")
            else:
                _ok(sf.setNodeSoil(i, 0, 0), "soil")
    assert sf.setNodeLink(0, n + 3, int(LinkType.Up), 1.0) == 1              # IndexError
    assert sf.setNodeLink(0, 1, 0, 1.0) == 6                                 # NoLink -> ParameterError
    assert sf.setNodeSoil(0, 0, 0) == 1                                      # surface node -> IndexError
    assert sf.setNodeSurface(ncol, 0) == 1                                   # soil node -> IndexError
    assert sf.setNodeSoil(ncol, 7, 0) == 6                                   # unknown soil -> ParameterError
    assert sf.setNodePond(ncol, 0.1) == 1
    _ok(sf.setHydraulicProperties(int(WRCModel.ModifiedVanGenuchten), int(MeanType.Logarithmic), 10.0), "hyd")
    assert sf.setHydraulicProperties(1, 2, 1000.0) == 6
    _ok(sf.setNumericalParameters(1.0, 600.0, 100, 10, 10, 4), "num")
    sf.setThreadsNumber(threads)
    for i in range(n):
        if i < ns:
            _ok(sf.setNodeWaterContent(i, 0.001), "wc")
        elif i < 2 * ns:
            _ok(sf.setNodeDegreeOfSaturation(i, 0.6), "se")
        elif i < 3 * ns:
            _ok(sf.setNodeWaterContent(i, 0.25), "wc")
        else:
            _ok(sf.setNodeMatricPotential(i, -1.5), "psi")
    assert sf.setNodeWaterContent(ncol, 1.5) == 6 and sf.setNodeDegreeOfSaturation(0, 0.5) == 1
    _ok(sf.initializeBalance(), "balance")
    getters = []
    for i in (0, ncol, n - 1):
        getters += [sf.getNodeWaterContent(i), sf.getNodeMaximumWaterContent(i), sf.getNodeMinimumWaterContent(i),
                    sf.getNodeAvailableWaterContent(i), sf.getNodeWaterDeficit(i, 3.0), sf.getNodeDegreeOfSaturation(i),
                    sf.getNodeWaterConductivity(i), sf.getNodeMatricPotential(i), sf.getNodeTotalPotential(i),
                    sf.getNodePond(i), sf.getNodeBoundaryWaterFlow(i)]
    getters += [sf.getNodeWaterContent(n + 5), sf.getNodePond(n)]                      # index sentinels
    dts = []
    for mm in (30.0, 0.0):
        for c in range(ncol):
            _ok(sf.setNodeWaterSinkSource(c, area * mm / 1000.0 / 3600.0), "sink")
        sf.computePeriod(3600.0)
    for i in range(2 * ncol, n):        # soil-soil links only (see compare(): stale-slot quirk Q2)
        getters += [sf.getNodeMaxWaterFlow(i, 1), sf.getNodeMaxWaterFlow(i, 2), sf.getNodeMaxWaterFlow(i, 3),
                    sf.getNodeSumLateralWaterFlowIn(i), sf.getNodeSumLateralWaterFlowOut(i)]
    out = snapshot(sf, n, dts)
    out["getters"] = np.array(getters)
    out["water_mbr"] = np.float64(sf.getWaterMBR())
    return out


SCENARIOS = {
    "storm": storm,
    "van_genuchten_geometric": van_genuchten_geometric,
    "evaporation_after_rain": evaporation_after_rain,
    "prescribed_and_urban": prescribed_and_urban,
    "saturated_bottom": saturated_bottom,
    "twenty_layers_saturated_mix": twenty_layers_saturated_mix,
    "dry_no_forcing": dry_no_forcing,
    "ragged_raster": ragged_raster,
    "config1_bundled_catchment": config1_bundled_catchment,
    "scalar_api_column": scalar_api_column,
    "raster_forcing_and_maps": raster_forcing_and_maps,
}
HEAT_SCENARIOS = {
    "heat_coupled": heat_coupled,
    "heat_diffusive_only": heat_diffusive_only,
    "heat_advective_column": heat_advective_column,
    "heat_advective_slope": heat_advective_slope,
}


# Per-scenario additions to the stated tolerances.  Accumulated link flows are sums of A'_ij (H_i - H_j) dt: they
# resolve head DIFFERENCES, so a trajectory on which the two sides' heads differ by d metres can differ by
# ~d * sum(dt) in a link flow sum although every head agrees to 1e-6 relative.  On the water scenarios the product's
# heads agree with the reference's to ~1e-11 m and no allowance is needed.  The advective slope case follows the
# reference's own runaway (SURVEY Q1): temperatures grow exponentially and amplify the 1-ulp differences between
# glibc's and CUDA's exp / log (measured with the product's power function on the host: |dH| 4e-9 m, |dT| 1.5e-5 K,
# link flows 9e-8 m3 of 7e-3), so its link flows get the allowance of a 2e-9 m head difference.
TOLERANCES = {
    "heat_advective_slope": dict(flow_head_tol=2e-9),
    "heat_advective_column": dict(flow_head_tol=2e-9),
}


def assert_bit_identical(a: dict, b: dict, what: str):
    """the same quantities, equal bit for bit (NaN equal to NaN)"""
    assert set(a) == set(b), what
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), f"{what}: {k} differs"


def assert_lockstep(a: dict, b: dict, psi):
    """Snapshots after ONE computeStep from the same state: the same accepted dt and approximation count,
    |dH| <= 1e-9 * max(1, |psi|) with psi the checker's matric potential after the step, and |dtheta| <= 1e-10
    on the soil nodes."""
    assert np.array_equal(a["dts"], b["dts"]), "accepted dt"
    assert a["counters"][0] == b["counters"][0], "approximation count"
    assert np.max(np.abs(a["TOTAL_POTENTIAL"] - b["TOTAL_POTENTIAL"]) / np.maximum(1.0, np.abs(psi))) <= 1e-9
    ns = int(b["n_surface"])
    assert np.max(np.abs(a["WATER_CONTENT"][ns:] - b["WATER_CONTENT"][ns:])) <= 1e-10


def compare(a: dict, b: dict, *, exact: bool, h_rel=1e-6, theta_abs=1e-7, flow_rel=1e-6, flow_head_tol=0.0,
            h_abs=None, totals_rel=None, sweeps=False, mbe_abs=None):
    """exact: bit-identical (oracle restatement vs reference, same libm).  Otherwise the fp64
    tolerances stated in tests/test_gpu_parity.py.  Off unless given: an absolute head bound h_abs [m], a
    relative bound totals_rel for the boundary totals other than flow_rel, equal sweep counts, and a bound
    mbe_abs [m3] on the difference of the last step's mass-balance errors (it scales with the rain)."""
    if exact:
        assert_bit_identical(a, b, "exact")
        return
    assert set(a) == set(b)
    first = next((k for k, (x, y) in enumerate(zip(a["dts"], b["dts"])) if x != y), None)
    assert np.array_equal(a["dts"], b["dts"]), f"accepted time-step sequences differ from step {first}"
    assert a["counters"][0] == b["counters"][0], "approximation count"
    if sweeps:
        assert a["counters"][1] == b["counters"][1], "sweep count"
    H, Hb = a["TOTAL_POTENTIAL"], b["TOTAL_POTENTIAL"]
    assert np.max(np.abs(H - Hb) / np.maximum(1.0, np.abs(Hb))) <= h_rel
    if h_abs is not None:
        assert np.max(np.abs(H - Hb)) <= h_abs, "total potential, absolute"
    assert np.max(np.abs(a["WATER_CONTENT"] - b["WATER_CONTENT"])) <= theta_abs
    assert np.max(np.abs(a["DEGREE_OF_SATURATION"] - b["DEGREE_OF_SATURATION"])) <= 1e-6
    K, Kb = a["WATER_CONDUCTIVITY"], b["WATER_CONDUCTIVITY"]
    assert np.all(np.abs(K - Kb) <= 1e-6 * np.abs(Kb) + 1e-18)
    # Link flow sums: a link whose conductance was 0 at an accepted step makes the reference read a
    # stale matrix slot (cpusolver.h:46-51, SURVEY Appendix B Q2); the product adds 0 for it.  Only
    # runoff (surface-surface) and infiltration (surface-soil) conductances can be 0, so link flows
    # are compared on soil-soil links: Up from the second soil layer on, Down and Lateral on soil nodes.
    ns = int(b["n_surface"])
    assert int(a["n_surface"]) == ns
    for k, first in (("BOUNDARY_WATER_FLOW", 0), ("MAX_FLOW_UP", 2 * ns), ("MAX_FLOW_DOWN", ns), ("SUM_LATERAL_FLOW", ns)):
        x, y = a[k][first:], b[k][first:]
        if x.size == 0:
            continue
        scale = max(1e-12, float(np.max(np.abs(y))))
        assert np.max(np.abs(x - y)) <= flow_rel * scale + 1e-12 + flow_head_tol * float(np.sum(b["dts"])), k
    assert a["total_water"] == np.float64(b["total_water"]) or abs(a["total_water"] - b["total_water"]) <= 1e-9 * abs(b["total_water"])
    bt, btb = a["boundary_totals"], b["boundary_totals"]
    assert np.all(np.abs(bt - btb) <= (flow_rel if totals_rel is None else totals_rel) * np.abs(btb) + 1e-12), "boundary totals"
    if mbe_abs is not None:
        assert abs(a["mbe_mbr"][0] - b["mbe_mbr"][0]) <= mbe_abs, "mass-balance error of the last step"
    if "TEMPERATURE" in a:
        # heat: the product iterates Jacobi where the reference sweeps Gauss-Seidel (same fixed point,
        # stopping tolerance 1e-10 K on the update); temperatures rel 1e-6, boundary diagnostics rel 1e-5
        T, Tb = a["TEMPERATURE"], b["TEMPERATURE"]
        assert np.max(np.abs(T - Tb) / np.maximum(1.0, np.abs(Tb))) <= 1e-6
        assert a["heat_counters"][0] == b["heat_counters"][0], "accepted heat sub-steps"
        # Q6: Jacobi (product) and Gauss-Seidel (reference) share the fixed point; the comparison is only
        # meaningful when both reached the tolerance in every heat solve, so that is asserted, not assumed
        assert b["heat_cap_hits"] == 0, "the reference's Gauss-Seidel stopped at its cap: trajectory is sweep dependent"
        assert a["heat_cap_hits"] == 0, "the product's heat solve stopped at its sweep cap"
        hb, hbb = a["heat_boundary"], b["heat_boundary"]
        assert np.all(np.abs(hb - hbb) <= 1e-5 * np.abs(hbb) + 1e-9)
        f, fb = a["heat_flux_down"], b["heat_flux_down"]
        assert np.all(np.abs(f - fb) <= 1e-4 * np.abs(fb) + 1e-3)          # float-rounded accumulations (heat.cpp:203-206)
    if "heat_advective_boundary" in a:
        # advective boundary flux [W m-2] of the HeatSurface and bottom nodes (heat.cpp:273-287, 302-309)
        g, gb = a["heat_advective_boundary"], b["heat_advective_boundary"]
        assert np.all(np.abs(g - gb) <= 1e-5 * np.abs(gb) + 1e-9)
        assert np.any((gb != 0.0) & (gb > -1000.0)), "the advective boundary term was never exercised"
    if "heat_flux_types" in a:
        # save mode All: one column per fluxTypes_t; float-rounded like heat_flux_down.  The advective column
        # (type 4) must be populated, or computeAdvectiveFlux did not run.
        f, fb = a["heat_flux_types"], b["heat_flux_types"]
        assert np.all(np.abs(f - fb) <= 1e-4 * np.abs(fb) + 1e-3 * (np.abs(fb) > 1.0) + 1e-12)
        assert np.all(np.abs(fb[:, 4]) > 0.0)
    if "rasters" in a:
        # float32 output maps: same NODATA cells, values within float rounding of the fp64 tolerance
        r, rb = a["rasters"], b["rasters"]
        assert np.array_equal(r == -9999.0, rb == -9999.0)
        assert np.all(np.abs(r - rb) <= 2e-6 * np.abs(rb) + 1e-7)
    if "getters" in a:
        g, gb = a["getters"], b["getters"]
        assert np.all(np.abs(g - gb) <= 1e-6 * np.abs(gb) + 1e-12)
