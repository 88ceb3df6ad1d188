"""GPU: parity on a 128 x 128 x (1+10) window of the C2 generator (180 224 nodes) over two storm hours against the
unmodified reference on all host cores: identical accepted-dt sequence, approximation and sweep counts, potentials,
water contents, link and boundary flow sums and the step's mass-balance error.  (Round 1 ran this as a script on a 256 x 256
window -- profiles/r01_parity_large.json; `python tests/validate_large.py 256 256 10 3` still does.)"""
import numpy as np
import pytest

from criteria3d_b200.synth import STORM_MM_H, Catchment, run_hours, setup
from scenarios import compare, snapshot

pytestmark = pytest.mark.gpu


def test_c2_window_two_storm_hours(product, checker):
    cat = Catchment(128, 128, 10)
    mm = STORM_MM_H[1:3]                   # 20 and 40 mm/h
    res = {}
    for name, sf in (("gpu", product), ("ref", checker)):
        setup(sf, cat, threads=0)          # reference: all host cores
        res[name] = snapshot(sf, cat.n_nodes, run_hours(sf, cat, mm))
    g, r = res["gpu"], res["ref"]
    assert len(g["dts"]) > 150, "the window is expected to need a few hundred accepted steps"
    sink_total = sum(np.sum(np.abs(cat.rain_sink_source(m))) * 3600.0 for m in mm)
    compare(g, r, exact=False, sweeps=True, mbe_abs=1e-6 * sink_total)
    approximations, sweeps = (int(v) for v in g["counters"])
    print(f"[c2 window] {len(g['dts'])} accepted steps, {approximations} approximations, {sweeps} sweeps on both sides; "
          f"max |dH| {np.max(np.abs(g['TOTAL_POTENTIAL'] - r['TOTAL_POTENTIAL'])):.2e} m, "
          f"max |dtheta| {np.max(np.abs(g['WATER_CONTENT'] - r['WATER_CONTENT'])):.2e}")
