"""CPU: the bounds of scenarios.compare() and scenarios.assert_lockstep(), one quantity at a time.  An oracle snapshot of a
small storm is compared with a copy of itself in which one quantity moved by just under the bound that covers it (must
pass) and by just over it (must fail), so a check that goes missing or a bound that goes slack fails here."""
import numpy as np
import pytest

from criteria3d_b200 import Field, SoilFluxes3D
from oracle import ORACLE_LIB
from scenarios import assert_lockstep, compare, storm

pytestmark = pytest.mark.skipif(not ORACLE_LIB.exists(), reason="needs oracle/libsf3d_oracle.so")


@pytest.fixture(scope="module")
def run():
    """the snapshot after 15 accepted steps of a 12 x 10 x (1+4) storm, and the matric potential then"""
    sf = SoilFluxes3D(ORACLE_LIB)
    ref = storm(sf, shape=(12, 10, 4), hours=(20.0,), max_steps=15)
    return ref, sf.get_field(Field.MATRIC_POTENTIAL, 0, ref["TOTAL_POTENTIAL"].size)


def _moved(ref, key, i, delta):
    out = dict(ref)
    out[key] = np.array(ref[key], copy=True)
    out[key][i] += delta
    return out


def _probe(ref, key, i, bound, check=None, **kw):
    """ref with ref[key][i] moved by just under `bound` passes `check` (default: compare with keywords kw), moved by
    just over it fails"""
    check = check or (lambda a: compare(a, ref, exact=False, **kw))
    check(_moved(ref, key, i, (1 - 1e-3) * bound))
    with pytest.raises(AssertionError):
        check(_moved(ref, key, i, (1 + 1e-3) * bound))


def test_state_bounds(run):
    ref, _ = run
    H, K = ref["TOTAL_POTENTIAL"], ref["WATER_CONDUCTIVITY"]
    i, k = int(np.argmax(np.abs(H))), int(np.argmax(K))
    _probe(ref, "TOTAL_POTENTIAL", i, 1e-6 * max(1.0, abs(H[i])))
    _probe(ref, "TOTAL_POTENTIAL", i, 1e-7, h_abs=1e-7)
    _probe(ref, "WATER_CONTENT", 0, 1e-7)
    _probe(ref, "WATER_CONTENT", 0, 1e-9, theta_abs=1e-9)
    _probe(ref, "DEGREE_OF_SATURATION", 0, 1e-6)
    _probe(ref, "WATER_CONDUCTIVITY", k, 1e-6 * K[k] + 1e-18)


@pytest.mark.parametrize("key,first_layer", [("BOUNDARY_WATER_FLOW", 0), ("MAX_FLOW_UP", 2), ("MAX_FLOW_DOWN", 1),
                                             ("SUM_LATERAL_FLOW", 1)])
def test_link_flow_bounds(run, key, first_layer):
    ref, _ = run
    first = first_layer * int(ref["n_surface"])
    j = first + int(np.argmax(np.abs(ref[key][first:])))
    _probe(ref, key, j, 1e-6 * abs(ref[key][j]) + 1e-12)


@pytest.mark.parametrize("j", range(4))
def test_boundary_total_bounds(run, j):
    ref, _ = run
    b = abs(ref["boundary_totals"][j])
    _probe(ref, "boundary_totals", j, 1e-6 * b + 1e-12)
    _probe(ref, "boundary_totals", j, 1e-9 * b + 1e-12, totals_rel=1e-9)


def test_total_water_and_mass_balance_error_bounds(run):
    ref, _ = run
    _probe(ref, "total_water", (), 1e-9 * abs(ref["total_water"]))
    _probe(ref, "mbe_mbr", 0, 1e-6, mbe_abs=1e-6)
    compare(_moved(ref, "mbe_mbr", 0, 1.0), ref, exact=False)                      # off unless a bound is given


def test_time_steps_and_counts_are_exact(run):
    ref, _ = run
    with pytest.raises(AssertionError, match="from step 3"):
        compare(_moved(ref, "dts", 3, np.spacing(ref["dts"][3])), ref, exact=False)
    with pytest.raises(AssertionError, match="approximation count"):
        compare(_moved(ref, "counters", 0, 1.0), ref, exact=False)
    compare(_moved(ref, "counters", 1, 1.0), ref, exact=False)                     # sweeps: off unless asked for
    compare(ref, ref, exact=False, sweeps=True)
    with pytest.raises(AssertionError, match="sweep count"):
        compare(_moved(ref, "counters", 1, 1.0), ref, exact=False, sweeps=True)


def test_lockstep_bounds(run):
    ref, psi = run

    def lockstep(a):
        assert_lockstep(a, ref, psi)
    i, ns = int(np.argmax(np.abs(psi))), int(ref["n_surface"])
    assert abs(psi[i]) > 1.0                                                       # the bound scales with |psi| there
    _probe(ref, "TOTAL_POTENTIAL", i, 1e-9 * abs(psi[i]), check=lockstep)
    _probe(ref, "WATER_CONTENT", ns, 1e-10, check=lockstep)
    for key, delta in (("dts", np.spacing(ref["dts"][0])), ("counters", 1.0)):
        with pytest.raises(AssertionError):
            lockstep(_moved(ref, key, 0, delta))
