"""Parity of the CUDA path (through the C ABI) with the oracle on identical inputs.

Tolerances (fp64; the only arithmetic differences are CUDA libm vs glibc and reduction order), applied by
scenarios.assert_lockstep and scenarios.compare:
  lock-step single computeStep : |dH| <= 1e-9 * max(1, |psi|), soil |dtheta| <= 1e-10, same accepted dt,
                                 same approximation count
  trajectory (hours of storm)  : same accepted-dt sequence and approximation count, |dH| <= 1e-6 * max(1, |H|),
                                 |dtheta| <= 1e-7, |dSe| <= 1e-6, K rel 1e-6, link flow sums within 1e-6 of the
                                 largest, boundary flow sums rel 1e-6 (+1e-12), total water rel 1e-9, the last
                                 step's mass-balance error within 1e-6 of the rain volume (sum|sink| x duration)
  integer maps                 : bit-exact
"""
import numpy as np
import pytest

from criteria3d_b200 import Field
from criteria3d_b200.synth import Catchment, run_hours, setup
from scenarios import assert_bit_identical, assert_lockstep, compare, heat_coupled, snapshot

pytestmark = pytest.mark.gpu


def _both(product, checker, cat, **kw):
    for sf in (product, checker):
        setup(sf, cat, **kw)


def test_index_maps_bit_exact(product, checker):
    cat = Catchment(37, 29, 5)
    _both(product, checker, cat)
    for slot in range(10):
        a, b = product.link_table(slot, 0, cat.n_nodes), checker.link_table(slot, 0, cat.n_nodes)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), f"slot {slot}"
        assert np.array_equal(a[2], b[2]), f"slot {slot} areas"
    for x, y in zip(product.node_meta(0, cat.n_nodes), checker.node_meta(0, cat.n_nodes)):
        assert np.array_equal(x, y)


def test_initial_state_and_storage(product, checker):
    cat = Catchment(32, 32, 6)
    _both(product, checker, cat)
    for f in (Field.TOTAL_POTENTIAL, Field.DEGREE_OF_SATURATION, Field.WATER_CONDUCTIVITY, Field.WATER_CONTENT):
        a, b = product.get_field(f, 0, cat.n_nodes), checker.get_field(f, 0, cat.n_nodes)
        assert np.allclose(a, b, rtol=1e-12, atol=1e-14), f.name
    assert product.getTotalWaterContent() == pytest.approx(checker.getTotalWaterContent(), rel=1e-12)


def test_lockstep_single_step(product, checker):
    cat = Catchment(40, 32, 6)
    _both(product, checker, cat)
    a, b = (snapshot(sf, cat.n_nodes, run_hours(sf, cat, [20.0], max_steps=1)) for sf in (product, checker))
    assert_lockstep(a, b, checker.get_field(Field.MATRIC_POTENTIAL, 0, cat.n_nodes))


@pytest.mark.parametrize("shape,hours", [((40, 32, 6), [20.0, 40.0, 5.0]), ((64, 48, 10), [40.0, 25.0])])
def test_trajectory(product, checker, shape, hours):
    cat = Catchment(*shape)
    _both(product, checker, cat)
    a, b = (snapshot(sf, cat.n_nodes, run_hours(sf, cat, hours)) for sf in (product, checker))
    sink_total = sum(np.sum(np.abs(cat.rain_sink_source(mm))) * 3600.0 for mm in hours)
    compare(a, b, exact=False, mbe_abs=1e-6 * sink_total)


def _storm_25_steps(sf):
    cat = Catchment(33, 27, 5)
    setup(sf, cat)
    return snapshot(sf, cat.n_nodes, run_hours(sf, cat, [30.0], max_steps=25))


def test_pattern_compressed_indices_are_bit_identical(product, checker, monkeypatch):
    """The sweeps read the column indices through 16-bit link patterns (2 B/node instead of 40 B).
    The map is verified on the device at finalize; forcing the explicit index array must give
    bit-identical results (integer work: exact), for the water sweep and for the heat sweep."""
    for name, scenario in (("water", _storm_25_steps), ("heat", heat_coupled)):
        runs = []
        for explicit in (False, True):
            if explicit:
                monkeypatch.setenv("SF3D_EXPLICIT_INDEX", "1")
            else:
                monkeypatch.delenv("SF3D_EXPLICIT_INDEX", raising=False)
            runs.append(scenario(product))
        assert_bit_identical(runs[0], runs[1], f"{name}: explicit vs pattern-compressed indices")
