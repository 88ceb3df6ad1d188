"""CPU: the C restatement (oracle/libsf3d_oracle.so) must be BIT-IDENTICAL to the unmodified
reference on every scenario, with one OpenMP thread on both sides.  This is what pins the oracle.
The reference is run live where its library is built (oracle/_ref/libsf3d_ref.so, `make -C oracle
ref`); elsewhere its stored outputs of the same scenarios stand in for it
(tests/golden/<scenario>.npz, written by tests/golden/make_golden.py from that library)."""
from pathlib import Path

import numpy as np
import pytest

from criteria3d_b200 import SoilFluxes3D
from oracle import ORACLE_LIB, REFERENCE_LIB
from scenarios import HEAT_SCENARIOS, SCENARIOS, compare

ALL = {**SCENARIOS, **HEAT_SCENARIOS}
GOLDEN = Path(__file__).parent / "golden"

pytestmark = pytest.mark.skipif(not ORACLE_LIB.exists(), reason="needs oracle/libsf3d_oracle.so")


@pytest.fixture(scope="module")
def libs():
    return SoilFluxes3D(ORACLE_LIB), (SoilFluxes3D(REFERENCE_LIB) if REFERENCE_LIB.exists() else None)


def _reference_outputs(ref, name):
    if ref is not None:
        return ALL[name](ref)
    with np.load(GOLDEN / f"{name}.npz") as z:
        return {k: z[k] for k in z.files}


@pytest.mark.parametrize("name", sorted(ALL))
def test_bit_identical(libs, name):
    port, ref = libs
    a = ALL[name](port)
    b = _reference_outputs(ref, name)
    compare(a, b, exact=True)


def test_thread_count_only_changes_reduction_bits(libs):
    """4 OpenMP threads vs 1: same accepted steps; potentials within 1e-9 (SURVEY 8c caveat i)."""
    port, _ = libs
    a = SCENARIOS["storm"](port, threads=1)
    b = SCENARIOS["storm"](port, threads=4)
    assert np.array_equal(a["dts"], b["dts"])
    assert np.max(np.abs(a["TOTAL_POTENTIAL"] - b["TOTAL_POTENTIAL"])) < 1e-9
