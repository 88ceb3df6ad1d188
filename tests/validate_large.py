"""One-off parity run on a larger window of the C2 generator (not collected by pytest: minutes of CPU
time for the reference).  Writes gpurun_out/parity_large.json.

    python tests/validate_large.py [rows cols soil_layers hours]
"""
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from criteria3d_b200 import SoilFluxes3D, load_product  # noqa: E402
from oracle import ORACLE_LIB, REFERENCE_LIB  # noqa: E402
from criteria3d_b200.synth import STORM_MM_H, Catchment, run_hours, setup  # noqa: E402
from scenarios import snapshot  # noqa: E402


def main():
    a = [int(x) for x in sys.argv[1:5]] + [256, 256, 10, 3][len(sys.argv) - 1:]
    rows, cols, layers, hours = a[:4]
    cat = Catchment(rows, cols, layers)
    mm = STORM_MM_H[1:1 + hours]
    gpu = load_product()
    chk = SoilFluxes3D(REFERENCE_LIB if REFERENCE_LIB.exists() else ORACLE_LIB)
    res, wall = {}, {}
    for name, sf in (("gpu", gpu), ("oracle", chk)):
        setup(sf, cat, threads=0)
        t0 = time.perf_counter()
        dts = run_hours(sf, cat, mm)
        wall[name] = time.perf_counter() - t0
        res[name] = snapshot(sf, cat.n_nodes, dts)
    g, o = res["gpu"], res["oracle"]
    out = {
        "grid": f"{rows}x{cols}x(1+{layers})", "nodes": cat.n_nodes, "hours_mm": mm, "checker": chk.backend,
        "accepted_steps": [len(g["dts"]), len(o["dts"])], "dt_sequences_identical": bool(np.array_equal(g["dts"], o["dts"])),
        "first_divergent_step": next((k for k, (x, y) in enumerate(zip(g["dts"], o["dts"])) if x != y), None),
        "approximations": [int(g["counters"][0]), int(o["counters"][0])], "sweeps": [int(g["counters"][1]), int(o["counters"][1])],
        "max_abs_dH": float(np.max(np.abs(g["TOTAL_POTENTIAL"] - o["TOTAL_POTENTIAL"]))),
        "max_abs_dtheta": float(np.max(np.abs(g["WATER_CONTENT"] - o["WATER_CONTENT"]))),
        "total_water": [float(g["total_water"]), float(o["total_water"])],
        # runoff, free and free lateral drainage, as in profiles/r01_parity_large.json
        "boundary_totals": [g["boundary_totals"][:3].tolist(), o["boundary_totals"][:3].tolist()],
        "mbe": [float(g["mbe_mbr"][0]), float(o["mbe_mbr"][0])], "wall_s": [wall["gpu"], wall["oracle"]],
    }
    Path(ROOT / "gpurun_out").mkdir(exist_ok=True)
    (ROOT / "gpurun_out" / "parity_large.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
