"""GPU: the -DSF3D_REFERENCE_ROUNDING build of the product (criteria3d_b200/libsf3d_b200_refround.so: pow() instead of
exp(y log x), area / distance and Math::computeMean evaluated per link as the reference writes them).  The DEFAULT build
is tolerance-parity: its few-ulp arithmetic differences could in principle flip one of the control loop's threshold tests
(Courant < 1.01, MBR < threshold, norm > 10 x best) on a long run and change the accepted-dt sequence from there on; no
such flip has been observed (tests/test_gpu_large_window.py, bench.py's accepted_dt against the reference arm, the 24 h
config-1 run), and this variant is the one to use when a caller needs the decision sequence itself pinned.  It is held
to the same lock-step test with TIGHTER state tolerances."""
from pathlib import Path

import numpy as np
import pytest

from criteria3d_b200 import SoilFluxes3D
from criteria3d_b200.synth import STORM_MM_H, Catchment, run_hours, setup
from scenarios import compare, snapshot

pytestmark = pytest.mark.gpu
LIB = Path(__file__).resolve().parent.parent / "criteria3d_b200" / "libsf3d_b200_refround.so"


def test_reference_rounding_build_lockstep_over_two_storm_hours(checker):
    if not LIB.exists():
        pytest.fail(f"{LIB} missing: run __graft_entry__.build()")
    sf = SoilFluxes3D(LIB)
    assert sf.backend == "b200"
    cat = Catchment(96, 96, 10)
    mm = STORM_MM_H[1:3]
    res = {}
    for name, lib in (("gpu", sf), ("ref", checker)):
        setup(lib, cat, threads=0)
        res[name] = snapshot(lib, cat.n_nodes, run_hours(lib, cat, mm))
    g, r = res["gpu"], res["ref"]
    # heads absolute in metres: ~230 m, so the default build's 1e-6 relative is 2e-4 m; measured 2.4e-8
    compare(g, r, exact=False, sweeps=True, h_abs=1e-7, theta_abs=1e-9, totals_rel=1e-9)
    print(f"[refround] {len(g['dts'])} steps, {int(g['counters'][1])} sweeps on both sides; "
          f"max |dH| {np.max(np.abs(g['TOTAL_POTENTIAL'] - r['TOTAL_POTENTIAL'])):.2e} m")
