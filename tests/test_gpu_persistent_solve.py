"""GPU: the persistent small-graph solve (all Jacobi sweeps of a solve in one cooperative launch, grid-wide barrier between
sweeps) against the launch-per-sweep path and against the reference.  Grid size, partial sums and fold order are the same
in both paths, so the residual norms -- and with them every decision and every potential -- must be BIT-identical between
the two; both are held to the usual tolerances against the reference."""
import os

import numpy as np
import pytest

from criteria3d_b200 import Field
from criteria3d_b200.synth import Catchment, run_hours, setup
from scenarios import SCENARIOS, assert_bit_identical, compare

pytestmark = pytest.mark.gpu


def _with_mode(mode, fn):
    old = os.environ.get("SF3D_PERSISTENT_SOLVE")
    if mode is None:
        os.environ.pop("SF3D_PERSISTENT_SOLVE", None)
    else:
        os.environ["SF3D_PERSISTENT_SOLVE"] = mode
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop("SF3D_PERSISTENT_SOLVE", None)
        else:
            os.environ["SF3D_PERSISTENT_SOLVE"] = old


@pytest.mark.parametrize("name", ["storm", "saturated_bottom", "config1_bundled_catchment", "twenty_layers_saturated_mix"])
def test_both_solve_paths_match_the_reference_and_each_other(product, checker, name):
    ref = SCENARIOS[name](checker)
    one = _with_mode(None, lambda: SCENARIOS[name](product))          # persistent (default for small graphs)
    per = _with_mode("0", lambda: SCENARIOS[name](product))           # one launch per sweep
    compare(one, ref, exact=False)
    compare(per, ref, exact=False)
    assert_bit_identical(one, per, f"{name}, persistent vs per sweep")


def test_launch_counts(product):
    """the persistent path needs one sweep launch per solve"""
    cat = Catchment(48, 40, 5)

    def run():
        setup(product, cat)
        c0 = product.counters()
        run_hours(product, cat, [20.0], max_steps=20)
        c1 = product.counters()
        return (c1["kernel_launches"] - c0["kernel_launches"], c1["sweeps"] - c0["sweeps"], c1["approximations"] - c0["approximations"],
                product.get_field(Field.TOTAL_POTENTIAL, 0, cat.n_nodes))
    l1, s1, a1, h1 = _with_mode(None, run)
    l0, s0, a0, h0 = _with_mode("0", run)
    assert (s1, a1) == (s0, a0) and np.array_equal(h1, h0)
    assert l1 < l0 - (s0 - a0) + 1, (l1, l0, s0, a0)          # at least (sweeps - solves) launches fewer
    print(f"[persistent solve] {s1} sweeps in {a1} solves: {l1} launches instead of {l0}")
