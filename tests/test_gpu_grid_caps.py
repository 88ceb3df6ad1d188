"""GPU: the kernels where a thread sweeps more than one row, against the reference.

Every kernel of sf3d_kernels.cu is a grid-stride loop over a capped grid of 256-thread blocks, and the last block
folds one partial per block in a fixed order.  The sweep, post, accept, begin-try, heat kernels and getters are
capped at 148 x 8 = 1184 blocks (more than one row per thread past 303 104 nodes), the node phase and the assembly
at 148 x 48 = 7104 blocks (past 1 818 624 nodes).  Every benchmark catchment is past both caps; the other
comparisons with the reference run far below them, with one row per thread and the persistent solve.

Small-grid build.  criteria3d_b200/libsf3d_b200_smallgrid.so is a TEST ARTEFACT that __graft_entry__.build() makes
from the product's sources with -DSF3D_MAX_BLOCKS=7 -DSF3D_WIDE_BLOCKS=3 (the caps are host-side launch sizes: its
device code is the product's).  On the 1-12 k node scenarios every kernel then loops over 1-15 rows per thread with
a ragged last pass, row loops carry their accumulators (Courant, norm, storage, the assembly's conductance scratch,
the ghost-row skips) from one row to the next, and the folds of 7 and 3 partials divide nothing.  Each scenario runs
with one launch per sweep and with the persistent solve, which must agree with the reference and bit for bit with
each other (same grid, same partials, same fold order: tests/test_gpu_persistent_solve.py).

Real caps.  The default product on both sides of the persistent-solve limit (N <= 303 104, DESIGN section 4) and on a
1.9 M node window past the wide cap, lock-step on the first step and over the first 20 accepted steps of a
40 mm/h hour; tolerances of tests/test_gpu_parity.py."""
import time
from pathlib import Path

import numpy as np
import pytest

from criteria3d_b200 import BoundaryType, Field, SoilFluxes3D
from criteria3d_b200.synth import Catchment, _ok, setup
from oracle import ORACLE_LIB
from scenarios import HEAT_SCENARIOS, SCENARIOS, TOLERANCES, compare, culvert_outlet
from test_gpu_parity import test_index_maps_bit_exact as _index_maps_bit_exact
from test_gpu_parity import test_pattern_compressed_indices_are_bit_identical as _pattern_indices_bit_identical
from test_gpu_persistent_solve import _with_mode

pytestmark = pytest.mark.gpu
SMALLGRID = Path(__file__).resolve().parent.parent / "criteria3d_b200" / "libsf3d_b200_smallgrid.so"
PERSISTENT_ALWAYS = "1000000000"        # SF3D_PERSISTENT_SOLVE: node limit of the persistent solve
CASES = {**SCENARIOS, **HEAT_SCENARIOS, "culvert_outlet": culvert_outlet}


@pytest.fixture(scope="module")
def smallgrid():
    if not SMALLGRID.exists():
        pytest.fail(f"{SMALLGRID} missing: run __graft_entry__.build()")
    sf = SoilFluxes3D(SMALLGRID)
    assert sf.backend == "b200"
    return sf


def _assert_bit_identical(a, b, what):
    for key in a:
        x, y = np.asarray(a[key]), np.asarray(b[key])
        if x.dtype.kind in "fiu" and x.shape == y.shape:
            assert np.array_equal(x, y, equal_nan=True), f"{what}: {key} differs between the two solve paths"


# ---- small-grid build ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_small_grid_both_solve_paths(smallgrid, checker, name):
    run = CASES[name]
    if name == "culvert_outlet":
        # the reference cannot run a culvert (SURVEY Q5): the C restatement is the checker, as in test_gpu_scenarios
        if not ORACLE_LIB.exists():
            pytest.skip("oracle library not built")
        ref = run(SoilFluxes3D(ORACLE_LIB))
        assert ref["culvert_total"] < 0.0
    else:
        ref = run(checker)
    out, launches = {}, {}
    for path, mode in (("per sweep", "0"), ("persistent", PERSISTENT_ALWAYS)):
        l0 = smallgrid.counters()["kernel_launches"]
        out[path] = _with_mode(mode, lambda: run(smallgrid))
        launches[path] = smallgrid.counters()["kernel_launches"] - l0
        compare(out[path], ref, exact=False, **TOLERANCES.get(name, {}))
        if "culvert_total" in ref:
            assert abs(out[path]["culvert_total"] - ref["culvert_total"]) <= 1e-6 * abs(ref["culvert_total"])
    _assert_bit_identical(out["persistent"], out["per sweep"], name)
    # the persistent solve is one launch per solve, the other path at least four (its first batch)
    assert launches["persistent"] < launches["per sweep"], launches
    approx, sweeps = (int(v) for v in out["persistent"]["counters"])
    print(f"[small grid] {name}: {len(ref['dts'])} steps, {approx} approximations, {sweeps} sweeps; launch per sweep "
          f"({launches['per sweep']} launches) and persistent solve ({launches['persistent']} launches) both match "
          f"the reference and agree bit for bit")


def test_small_grid_index_maps_bit_exact(smallgrid, checker):
    _index_maps_bit_exact(smallgrid, checker)


def test_small_grid_pattern_compressed_indices_are_bit_identical(smallgrid, checker, monkeypatch):
    _pattern_indices_bit_identical(smallgrid, checker, monkeypatch)


# ---- the real caps, default product ------------------------------------------------------------------------------
RAIN_MM_H = 40.0


def _first_steps_of_hour(sf, cat, steps=20):
    """setup on all host cores, then the first `steps` accepted steps of an hour of RAIN_MM_H.  Returns the state after
    the first step (lock-step comparison), the state after the last one, the kernel launches and the time spent in
    computeStep."""
    setup(sf, cat, threads=0)
    sink = np.zeros(cat.n_nodes)
    sink[: cat.n_surface] = cat.rain_sink_source(RAIN_MM_H)
    _ok(sf.set_field(Field.WATER_SINK_SOURCE, 0, sink), "sink")
    l0 = sf.counters()["kernel_launches"]
    t0 = time.perf_counter()
    dts = [sf.computeStep(3600.0)]
    wall = time.perf_counter() - t0
    first = dict(dt=dts[0], approximations=sf.counters()["approximations"],
                 H=sf.get_field(Field.TOTAL_POTENTIAL, 0, cat.n_nodes), W=sf.get_field(Field.WATER_CONTENT, 0, cat.n_nodes),
                 psi=sf.get_field(Field.MATRIC_POTENTIAL, 0, cat.n_nodes))
    t0 = time.perf_counter()
    while len(dts) < steps and sum(dts) < 3600.0:
        dts.append(sf.computeStep(3600.0 - sum(dts)))
    wall += time.perf_counter() - t0
    c = sf.counters()
    last = dict(dts=np.array(dts), H=sf.get_field(Field.TOTAL_POTENTIAL, 0, cat.n_nodes),
                W=sf.get_field(Field.WATER_CONTENT, 0, cat.n_nodes),
                boundary=np.array([sf.getTotalBoundaryWaterFlow(int(b)) for b in
                                   (BoundaryType.Runoff, BoundaryType.FreeDrainage, BoundaryType.FreeLateralDrainage)]),
                total_water=np.float64(sf.getTotalWaterContent()),
                counters=np.array([c["steps"], c["approximations"], c["sweeps"]]), last_mbe=np.float64(c["last_mbe"]))
    return dict(first=first, last=last, launches=c["kernel_launches"] - l0, wall=wall)


def _assert_matches_reference(cat, gpu, ref):
    f, fr = gpu["first"], ref["first"]
    # lock-step single step (test_gpu_parity.test_lockstep_single_step)
    assert f["dt"] == fr["dt"] and f["approximations"] == fr["approximations"], "first step"
    assert np.max(np.abs(f["H"] - fr["H"]) / np.maximum(1.0, np.abs(fr["psi"]))) <= 1e-9
    assert np.max(np.abs(f["W"] - fr["W"])[cat.n_surface:]) <= 1e-10
    # trajectory (test_gpu_parity.test_trajectory)
    l, lr = gpu["last"], ref["last"]
    first = next((k for k, (x, y) in enumerate(zip(l["dts"], lr["dts"])) if x != y), None)
    assert np.array_equal(l["dts"], lr["dts"]), f"accepted time-step sequences differ from step {first}"
    assert np.array_equal(l["counters"], lr["counters"]), "steps, approximations, sweeps"
    assert np.max(np.abs(l["H"] - lr["H"]) / np.maximum(1.0, np.abs(lr["H"]))) <= 1e-6
    assert np.max(np.abs(l["W"] - lr["W"])) <= 1e-7
    for a, b in zip(l["boundary"], lr["boundary"]):
        assert a == pytest.approx(b, rel=1e-6, abs=1e-9)
    assert l["total_water"] == pytest.approx(lr["total_water"], rel=1e-9)
    sink_total = np.sum(np.abs(cat.rain_sink_source(RAIN_MM_H))) * np.sum(lr["dts"])
    assert abs(l["last_mbe"] - lr["last_mbe"]) <= 1e-6 * sink_total


def _switch_catchment(n_nodes):
    if n_nodes == 303_104:
        return Catchment(148, 256, 7)                       # 148 x 256 x (1+7): one row per thread of 1184 blocks
    valid = np.ones((149, 256), bool)                       # eight nodes more: 37 889 cells x 8 layers
    valid[60:75, 100:117] = False                           # a 15 x 17 hole of NODATA cells
    return Catchment(149, 256, 7, valid=valid)


@pytest.mark.parametrize("n_nodes,persistent", [(303_104, True), (303_112, False)], ids=["at-limit", "past-limit"])
def test_persistent_switch_point(product, checker, n_nodes, persistent):
    cat = _switch_catchment(n_nodes)
    assert cat.n_nodes == n_nodes
    default = _with_mode(None, lambda: _first_steps_of_hour(product, cat))
    per_sweep = _with_mode("0", lambda: _first_steps_of_hour(product, cat))
    ref = _first_steps_of_hour(checker, cat)
    _assert_matches_reference(cat, default, ref)
    _assert_bit_identical(default["last"], per_sweep["last"], f"N={n_nodes}")
    l1, l0 = default["launches"], per_sweep["launches"]
    steps, approximations, sweeps = (int(v) for v in default["last"]["counters"])
    if persistent:      # at least (sweeps - solves) launches fewer (test_gpu_persistent_solve.test_launch_counts)
        assert l1 < l0 and l1 < l0 - (sweeps - approximations) + 1, \
            f"N={n_nodes}: the persistent solve did not run ({l1} launches, {l0} with one launch per sweep)"
    else:
        assert l1 == l0, f"N={n_nodes}: expected one launch per sweep ({l1} launches, {l0} with SF3D_PERSISTENT_SOLVE=0)"
    print(f"[switch point] N={n_nodes}: {'persistent solve' if l1 < l0 else 'one launch per sweep'} "
          f"({l1} launches; {l0} with one launch per sweep), {steps} steps, {sweeps} sweeps on both sides; "
          f"computeStep wall time: product {default['wall']:.2f} s, {checker.backend} {ref['wall']:.2f} s")


def test_past_the_wide_cap(product, checker):
    """416 x 416 x (1+10) = 1 903 616 nodes: node phase and assembly give some threads two rows, the sweep gives every
    thread 6-7 rows with a partial last pass, and the folds are of 1184 and 7104 partials"""
    cat = Catchment(416, 416, 10)
    assert cat.n_nodes == 1_903_616
    gpu = _first_steps_of_hour(product, cat)
    ref = _first_steps_of_hour(checker, cat)
    _assert_matches_reference(cat, gpu, ref)
    steps, approximations, sweeps = (int(v) for v in gpu["last"]["counters"])
    print(f"[wide cap] N={cat.n_nodes}: {steps} steps, {approximations} approximations, {sweeps} sweeps on both sides; "
          f"computeStep wall time: product {gpu['wall']:.2f} s, {checker.backend} {ref['wall']:.2f} s")
