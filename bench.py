#!/usr/bin/env python
"""bench.py -- node-iterations/s of the soilFluxes3D water time step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # the CUDA product (default N=1)
    python bench.py --impl reference --steps K --warmup W     # the reference's CPU/OpenMP path
    python bench.py ... --dump-outputs DIR                    # also write what the last timed step computed

--dump-outputs DIR writes, after the timed regions of the headline workload (rank 0's slab when N > 1), what a caller
of the timed path receives from its last step, one DIR/<name>.npy each: accepted_dt (float64, the computeStep return
values of the timed steps), matric_potential_maps (float32 [layers, rows, cols], the maps the e2e region downloads),
total_potential and water_content (float64 per node; temperature too with --heat).  An array larger than its cap is
replaced by the same seeded sample of its flattened values on every run: 56 MiB + 8 B per timed step at most.  The inputs are a
deterministic function of the arguments, so two builds run with the same arguments can be compared file by file.

A "step" is one computeStep() (soilFluxes3D.cpp:1785) = one accepted water time step of the
catchment: Picard approximations, each an assembly pass and a batch of Jacobi sweeps.  The
headline unit is node-iterations/s = nodes x Jacobi sweeps executed / time (SURVEY 8d); simulated
hours per wall second are reported beside it.

  value : inputs resident in HBM, device time (CUDA events on the library's stream, max over ranks)
  e2e   : the same metric on the SAME accepted steps (state saved after warm-up and restored before each timed
          region) through the C ABI with HOST buffers: every step uploads the forcing
          as the hourly precipitation map (sf3d_ext_set_forcing_rasters = assignPrecipitation +
          setSinkSource, pinned host memory) and reads back the matric potential maps of all
          layers (sf3d_ext_get_layer_rasters_async = computeCriteria3DMap per layer, as saveModelsState: the copy of
          step k overlaps the kernels of step k + 1 on a second stream, the host waits for it before the next one is
          issued and for the last one before the region ends); host<->device copies are inside the timed region
  roofline : Jacobi sweep kernel, algorithmic bytes (12 B per link + 32 B per node) / measured
          kernel time (CUDA events around every launch, in a third replay of the same steps: the events cost ~10 %
          of the step, so the value region runs without them) vs the measured HBM copy bandwidth of MEASURED_PEAKS.json
  cpu_baseline : the reference (oracle/_ref, unmodified sources) on the box's host cores: the full grid, the same
          warm-up and forcing, as many of the same steps as fit a wall-time budget
  parity_check (N > 1) : the N-rank slab path against the reference on a small whole catchment, before timing
  c4 : the same measurement on a C4 slab (512 x 4096 x (1+20) per GPU, lower third saturated); 8 slabs = configs[3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOAD = dict(rows=1024, cols=1024, soil_layers=10)          # BASELINE.json configs[1]
RAIN_MM_H = 40.0                                                # peak hour of the C2 hyetograph
# The CPU legs (reference arm and in-line cpu_baseline) run the FULL C2 grid on the same steps as the GPU arm (same
# generator, forcing and warm-up): 7.5 GB of reference state, ~2-3 s per computeStep on 16 cores; the timed part is
# bounded by a wall-time budget, the number of steps actually timed is reported.
C4_SLAB = dict(rows=512, cols=4096, soil_layers=20)            # per-GPU slab of BASELINE.json configs[3] (8 of them = 4096 x 4096)
DUMP_MAP_VALUES = 11 * 1024 * 1024                              # float32 map values kept by --dump-outputs: all 11 maps of C2 (44 MiB)
DUMP_NODE_VALUES = 1 << 19                                      # float64 node values kept per field (4 MiB)


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.device)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.split(",") for r in Path(self.path).read_text().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            out["sm_mhz"] = float(np.median(sm)) if sm else None
            out["sm_max_mhz"] = float(rows[0][2]) if rows else None
            out["power_w_max"] = max(float(r[3]) for r in rows) if rows else None
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            seen = set()
            for r in rows:
                for k, nme in enumerate(names):
                    if r[4 + k].strip().lower().startswith("active"):
                        seen.add(nme)
            out["reasons"] = sorted(seen)
            out["samples"] = len(rows)
        except Exception as e:  # noqa: BLE001
            out["error"] = str(e)
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out


def cpu_run(sample: dict, steps: int, warmup: int, budget_s: float):
    """Time the reference CPU implementation (all host threads) on the same steps the GPU arm times: the same
    generator, the same raster forcing, `warmup` untimed computeStep calls, then up to `steps` timed ones
    (bounded by budget_s seconds of wall time)."""
    from criteria3d_b200 import SoilFluxes3D
    from oracle import ORACLE_LIB, REFERENCE_LIB
    from criteria3d_b200.synth import Catchment, setup
    if REFERENCE_LIB.exists():
        sf, kind = SoilFluxes3D(REFERENCE_LIB), "reference"
    else:
        sf, kind = SoilFluxes3D(ORACLE_LIB), "port"
    cat = Catchment(sample["rows"], sample["cols"], sample["soil_layers"], saturated_bottom=sample.get("saturated_bottom", False))
    t_setup = time.perf_counter()
    setup(sf, cat, threads=0)
    cores = sf.setThreadsNumber(0)
    assert sf.set_forcing_rasters(precipitation=cat.rain_raster(RAIN_MM_H)) == 0
    t_setup = time.perf_counter() - t_setup
    for _ in range(warmup):
        sf.computeStep(3600.0)
    c0 = sf.counters()
    t0 = time.perf_counter()
    sim = 0.0
    done = 0
    dts = []
    for _ in range(steps):
        dts.append(sf.computeStep(3600.0))
        sim += dts[-1]
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    wall = time.perf_counter() - t0
    c1 = sf.counters()
    sweeps = c1["sweeps"] - c0["sweeps"]
    full = (sample["rows"], sample["cols"], sample["soil_layers"]) == (WORKLOAD["rows"], WORKLOAD["cols"], WORKLOAD["soil_layers"])
    return {
        "value": cat.n_nodes * sweeps / wall, "unit": "node-iterations/s", "cores": int(cores), "kind": kind,
        "sample": ("the full " if full else "a window of the same generator, ") + f"{sample['rows']}x{sample['cols']}x(1+{sample['soil_layers']}) grid, "
                  f"{warmup} warm-up + {done} timed computeStep calls" + ("" if done == steps else f" (of {steps}: {budget_s:.0f} s budget)")
                  + f", {sweeps} sweeps, {wall:.2f} s wall (setup {t_setup:.1f} s untimed)",
        "sim_hours_per_wall_s": sim / 3600.0 / wall, "ms_per_step": 1e3 * wall / max(done, 1),
        "steps": done, "sweeps": int(sweeps), "approximations": int(c1["approximations"] - c0["approximations"]),
        "n_nodes": cat.n_nodes, "accepted_dt": dts, "same_config": bool(full),
    }


def _seeded_sample(a: np.ndarray, cap: int, seed: int = 0) -> np.ndarray:
    """`a` itself when it has at most `cap` values, else `cap` of its flattened values at positions fixed by `seed`"""
    if a.size <= cap:
        return np.array(a)
    idx = np.sort(np.random.default_rng(seed).choice(a.size, cap, replace=False))
    return np.ascontiguousarray(a).reshape(-1)[idx]


def last_step_outputs(sf, N, dts, maps, heat) -> dict:
    """what a caller of the timed path holds after its last step (see --dump-outputs in the module docstring)"""
    from criteria3d_b200 import Field
    out = {"accepted_dt": np.asarray(dts, dtype=np.float64),
           "matric_potential_maps": _seeded_sample(maps, DUMP_MAP_VALUES)}
    fields = [("total_potential", Field.TOTAL_POTENTIAL), ("water_content", Field.WATER_CONTENT)]
    if heat:
        fields.append(("temperature", Field.TEMPERATURE))
    for name, f in fields:
        out[name] = _seeded_sample(sf.get_field(f, 0, N), DUMP_NODE_VALUES)
    return out


def config_name(args, world) -> str:
    """BASELINE.json configuration the shape corresponds to (C2 is the headline single-GPU workload)"""
    shape = (args.rows * world, args.cols, args.soil_layers)
    if args.heat and shape == (1024, 1024, 10):
        return "C3"
    return {(1024, 1024, 10): "C2", (4096, 4096, 20): "C4", (8192, 8192, 20): "C5"}.get(shape, "C2-like slab" if world > 1 else "custom")


def timed_region(sf, steps, stream, barrier, *, e2e=None):
    """`steps` computeStep calls between two CUDA events on the library's stream (barrier + synchronize on both
    sides).  e2e = (rain_np, out_np, cat, Field): every step also uploads the forcing raster from pinned host memory
    and downloads the matric-potential maps of all layers.  Returns (ms, wall_s, simulated_s, accepted_dt, host_ms)."""
    import torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tcall = [0.0, 0.0, 0.0]
    dts = []
    barrier()
    t0 = time.perf_counter()
    ev0.record(stream)
    checksum = 0.0
    for k in range(steps):
        ta = time.perf_counter()
        if e2e:
            rain_np, out_np, cat, Field = e2e
            sf.set_forcing_rasters(precipitation=rain_np)                  # H2D, rows x cols floats -> sink/source on the device
        tb = time.perf_counter()
        dts.append(sf.computeStep(3600.0))
        tc = time.perf_counter()
        if e2e:
            # D2H, layers x rows x cols floats into one of two page-locked buffers: the copy of step k runs on the library's
            # copy stream beside the kernels of step k + 1; the host waits for it (and reads the maps) before it hands the
            # other buffer to step k + 1
            sf.wait_rasters()
            if k > 0:
                checksum += float(out_np[(k - 1) & 1][0, 0, 0])
            sf.get_layer_rasters_async(Field.MATRIC_POTENTIAL, 0, cat.layers, (cat.rows, cat.cols), out_np[k & 1])
        td = time.perf_counter()
        tcall[0] += tb - ta; tcall[1] += tc - tb; tcall[2] += td - tc
    if e2e:
        te = time.perf_counter()
        sf.wait_rasters()                                    # the last step's maps are on the host before the region ends
        checksum += float(out_np[(steps - 1) & 1][0, 0, 0])
        tcall[2] += time.perf_counter() - te
    ev1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    return ev0.elapsed_time(ev1), wall, float(sum(dts)), dts, [1e3 * t / max(steps, 1) for t in tcall]


def run_workload(sf, args, shape, rank, local_rank, world, steps, warmup, *, heat=False, saturated_bottom=False, with_e2e=True,
                 keep_outputs=False):
    """Set up `shape` = (rows per GPU, cols, soil layers) on this rank (a row slab when world > 1), warm up, then time
    the SAME `steps` accepted steps twice from the same saved state: device-resident (value) and end to end through
    the C ABI with host buffers (e2e).  Returns this rank's measurements (times already max-reduced over ranks) and,
    with keep_outputs (needs with_e2e), what the last timed step computed under "outputs"."""
    import torch
    import torch.distributed as dist
    from criteria3d_b200 import Field
    from criteria3d_b200.synth import Catchment, setup
    rows, cols, layers = shape
    if world > 1:
        from criteria3d_b200.mgpu import setup_slab
        slab, cat = setup_slab(sf, rows * world, cols, layers, rank, world, saturated_bottom=saturated_bottom)
        n_owned = slab.n_owned
    else:
        cat = Catchment(rows, cols, layers, heat=heat, saturated_bottom=saturated_bottom)
        setup(sf, cat)
        n_owned = cat.n_nodes
    N = cat.n_nodes
    stream = torch.cuda.ExternalStream(sf.stream(), device=local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # forcing: the hourly precipitation map [mm h-1], float32 like the reference's meteo maps, from pinned host memory;
    # result: the matric potential maps of all layers, float32 rasters as saveModelsState / computeCriteria3DMap produce them
    rain_host = torch.from_numpy(cat.rain_raster(RAIN_MM_H)).pin_memory()
    rain_np = rain_host.numpy()
    out_host = [torch.empty((cat.layers, cat.rows, cat.cols), dtype=torch.float32).pin_memory() for _ in range(2)]
    out_np = [t.numpy() for t in out_host]
    assert sf.set_forcing_rasters(precipitation=rain_np) == 0
    for _ in range(warmup):
        sf.computeStep(3600.0)
    for b in range(2):                                    # untimed warm-up of the host-facing call (allocates both staging buffers)
        sf.get_layer_rasters_async(Field.MATRIC_POTENTIAL, 0, cat.layers, (cat.rows, cat.cols), out_np[b])
    sf.wait_rasters()

    # the state both timed regions start from (heat runs are not replayed: temperatures would need the same treatment)
    replay = not heat
    if replay:
        H0 = sf.get_field(Field.TOTAL_POTENTIAL, 0, N)
        dt0 = sf.counters()["delta_t_curr"]

        def restore():
            assert sf.set_field(Field.TOTAL_POTENTIAL, 0, H0) == 0
            assert sf.set_time_step(dt0) == 0
            assert sf.initializeBalance() == 0
        restore()

    # ---------------- timed region 1: inputs resident in HBM --------------------------------
    # Per-launch CUDA events (sf3d_ext_profile) cost ~10 % of a C2 step (two event records around each of ~32 launches per
    # step break the back-to-back launches), so the value region runs WITHOUT them; the kernel break-down comes from a third
    # replay of the same steps below.  Coupled-heat runs cannot be replayed and keep the events in this region.
    clocks = ClockSampler(local_rank)
    clocks.start()
    if not replay:
        sf.profile(True)
    c0 = sf.counters()
    ms, _wall, sim, dts, _ = timed_region(sf, steps, stream, barrier)
    c1 = sf.counters()
    ktimes, ms_prof = (sf.kernel_times(), ms) if not replay else (None, None)
    if not replay:
        sf.profile(False)
    res = {"cat": cat, "N": N, "n_owned": n_owned, "ms": ms, "sim": sim, "dts": dts, "c0": c0, "c1": c1,
           "sweeps": c1["sweeps"] - c0["sweeps"], "h2d": int(rain_np.nbytes), "d2h": int(out_np[0].nbytes), "replay": replay}

    # ---------------- timed region 2: the same steps end to end through the C ABI, host buffers ---------------
    if with_e2e:
        if replay:
            restore()
        ce0 = sf.counters()
        ms_e, wall_e, sim_e, dts_e, host_ms = timed_region(sf, steps, stream, barrier, e2e=(rain_np, out_np, cat, Field))
        ce1 = sf.counters()
        res.update({"ms_e2e": max(ms_e, wall_e * 1e3), "sim_e2e": sim_e, "sweeps_e2e": ce1["sweeps"] - ce0["sweeps"],
                    "host_ms": host_ms, "same_steps": bool(replay and dts_e == dts and (ce1["sweeps"] - ce0["sweeps"]) == res["sweeps"])})

    # ---------------- region 3: the same steps once more with per-launch CUDA events: kernel_ms, roofline ---------------
    if replay:
        restore()
        sf.profile(True)
        cp0 = sf.counters()
        ms_prof, _w, _s, dts_p, _ = timed_region(sf, steps, stream, barrier)
        cp1 = sf.counters()
        ktimes = sf.kernel_times()
        sf.profile(False)
        res["profiled_same_steps"] = bool(dts_p == dts and (cp1["sweeps"] - cp0["sweeps"]) == res["sweeps"])
    res["ktimes"], res["ms_profiled"] = ktimes, ms_prof
    res["clocks"] = clocks.stop()
    if keep_outputs:
        assert with_e2e and steps > 0, "the outputs of the last timed step are those of the e2e region"
        # the e2e region runs last among the timed ones (region 3 replays the same steps to the same state)
        res["outputs"] = last_step_outputs(sf, N, dts_e, out_np[(steps - 1) & 1], heat)

    # max over ranks of the device times; owned nodes summed (every rank executes the same sweeps on its slab)
    if world > 1:
        t = torch.tensor([res["ms"], res.get("ms_e2e", 0.0)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["ms"], res["ms_e2e"] = float(t[0]), float(t[1])
        owned = torch.tensor([float(n_owned)], dtype=torch.float64, device="cuda")
        dist.all_reduce(owned)
        res["owned_global"] = float(owned[0])
    else:
        res["owned_global"] = float(N)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=WORKLOAD["rows"])
    ap.add_argument("--cols", type=int, default=WORKLOAD["cols"])
    ap.add_argument("--soil-layers", type=int, default=WORKLOAD["soil_layers"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4-slab block (512 x 4096 x (1+20) per GPU)")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the N-rank slab-vs-reference parity check")
    ap.add_argument("--c4-steps", type=int, default=None, help="timed steps of the C4-slab block (default: --steps)")
    ap.add_argument("--saturated-bottom", action="store_true", help="config 4: lower third of the layers start saturated")
    ap.add_argument("--heat", action="store_true", help="config 3: coupled heat transport (not the headline workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.c4_steps is None:
        args.c4_steps = args.steps
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA product (--impl b200)")
    if args.dump_outputs is not None and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step (--steps >= 1)")
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return
        sample = dict(rows=args.rows, cols=args.cols, soil_layers=args.soil_layers, saturated_bottom=args.saturated_bottom)
        r = cpu_run(sample, args.steps, args.warmup, budget_s=150.0)
        line = {
            "impl": "reference", "metric": "node-iterations/s", "value": r["value"], "unit": "node-iterations/s",
            "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C2 synthetic {args.rows}x{args.cols} DEM x (1+{args.soil_layers}) layers, {RAIN_MM_H:g} mm/h storm hour, water only, "
                                   "Richards + Manning runoff (reference CPU/OpenMP path: " + r["sample"] + ")",
                       "same_config": r["same_config"]},
            "sim_hours_per_wall_s": r["sim_hours_per_wall_s"], "sweeps": r["sweeps"], "approximations": r["approximations"],
            "accepted_dt": r["accepted_dt"],
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "node-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), flush=True)
        return

    import torch
    import torch.distributed as dist
    from criteria3d_b200 import load_product

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sf = load_product()
    assert sf.set_device(local_rank) == 0
    parity = parity_c4 = None
    if world > 1:
        from criteria3d_b200.mgpu import wire_ranks
        wire_ranks(sf, rank, world)
        if not args.no_parity_check:
            # N-rank slab path against the reference on a small whole catchment, before anything is timed
            sys.path.insert(0, str(ROOT / "tests"))
            from mgpu_slab_check import reduce_over_ranks, slab_parity
            parity = reduce_over_ranks(slab_parity(sf, rank, world))
            # ... and the C4 recipe (20 soil layers, saturated lower third, free drainage) at small size
            parity_c4 = reduce_over_ranks(slab_parity(sf, rank, world, c4=True)) if not args.no_c4 else None

    # weak scaling: every GPU owns a rows x cols slab of a (world * rows) x cols catchment
    r = run_workload(sf, args, (args.rows, args.cols, args.soil_layers), rank, local_rank, world, args.steps, warmup,
                     heat=args.heat, saturated_bottom=args.saturated_bottom, keep_outputs=args.dump_outputs is not None and rank == 0)
    if "outputs" in r:
        args.dump_outputs.mkdir(parents=True, exist_ok=True)
        for name, a in r.pop("outputs").items():
            np.save(args.dump_outputs / f"{name}.npy", a)
    c4 = None
    headline_c2 = (args.rows, args.cols, args.soil_layers) == (WORKLOAD["rows"], WORKLOAD["cols"], WORKLOAD["soil_layers"]) and not args.heat
    if headline_c2 and not args.no_c4:
        c4 = run_workload(sf, args, (C4_SLAB["rows"], C4_SLAB["cols"], C4_SLAB["soil_layers"]), rank, local_rank, world,
                          args.c4_steps, 3, saturated_bottom=True, with_e2e=False)

    if rank == 0:
        peak, peak_src = measured_peak()
        cat, N, ms, ktimes, c0, c1 = r["cat"], r["N"], r["ms"], r["ktimes"], r["c0"], r["c1"]
        sweeps, sweeps_e2e = r["sweeps"], r["sweeps_e2e"]
        tot_iter, tot_iter_e2e = r["owned_global"] * float(sweeps), r["owned_global"] * float(sweeps_e2e)
        links = c1["links"]
        bytes_sweep = 12.0 * links + 32.0 * N
        bytes_repr = 8.0 * links + 34.0 * N         # what this representation must move: values + b, z, x in, x out + 2 B pattern id
        jac = ktimes["jacobi"]
        jac_s = jac["ms"] * 1e-3
        jac_gbs = bytes_sweep * sweeps / jac_s / 1e9 if jac["ms"] > 0 else None
        # assembly (node phase + link phase): SURVEY 8d algorithmic bytes 144 N + 12 Lk + 8 nnz per approximation
        approx = int(c1["approximations"] - c0["approximations"])
        bytes_asm = 144.0 * N + 12.0 * links + 8.0 * links
        asm_ms = ktimes["assemble"]["ms"] + ktimes["node_phase"]["ms"]
        asm_gbs = bytes_asm * approx / (asm_ms * 1e-3) / 1e9 if asm_ms > 0 and approx else None
        traffic = None
        tfile = ROOT / "profiles" / "jacobi_traffic.json"
        if tfile.exists():
            try:
                tj = json.loads(tfile.read_text())
                # the capture is of the C2 single-GPU shape; other shapes have no capture
                traffic = tj.get("dram_bytes_per_launch") if int(tj.get("nodes", 0)) == int(N) else None
            except Exception:
                traffic = None
        line = {
            "metric": "node-iterations/s", "value": tot_iter / (ms * 1e-3), "unit": "node-iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"{config_name(args, world)} synthetic {args.rows}x{args.cols} DEM per GPU x (1+{args.soil_layers}) layers, "
                            f"{RAIN_MM_H:g} mm/h storm hour, " + ("coupled heat (diffusive + latent)" if args.heat else "water only") + ", Richards + Manning runoff",
                "nodes_per_gpu": N, "links_per_gpu": int(links),
                "parallelism": "single GPU" if world == 1 else
                               f"{world} row slabs of {args.rows} DEM rows each (+1 ghost row per side); per sweep ONE kernel: boundary rows first, "
                               + ("stored into the neighbours' ghost rows over NVLink peer memory while the interior rows are swept, then the in-kernel "
                                  "mailbox all-reduce of the residual + stopping rule" if getattr(sf, "halo_mode", "nccl") == "peer-memory"
                                  else "ncclSend/ncclRecv halo of x + ncclAllReduce of the residual")
                               + f"; Courant / balance all-reduces inside the producing kernels; global catchment {args.rows * world}x{args.cols}",
                "l2": "working set per sweep (12 B/link + 32 B/node = %.2f GB) >> 126 MB L2; no explicit flush" % (bytes_sweep / 1e9),
                "numerics": "setNumericalParameters(0.5, 3600, 150, 10, 10, 3)",
                "timed_steps": "value and e2e time the SAME accepted steps: the state after warm-up (total potential, deltaTcurr) is saved and "
                               "restored (sf3d_ext_set_field + sf3d_ext_set_time_step + initializeBalance) before each region" if r["replay"] else
                               "consecutive steps (coupled heat runs are not replayed)",
            },
            "sim_hours_per_wall_s": r["sim"] / 3600.0 / (ms * 1e-3),
            "sweeps": int(sweeps), "approximations": approx,
            "heat_steps": int(c1["heat_steps"] - c0["heat_steps"]), "heat_sweeps": int(c1["heat_sweeps"] - c0["heat_sweeps"]),
            "heat_cap_hits": int(c1["heat_cap_hits"] - c0["heat_cap_hits"]),
            "tries": int(c1["tries"] - c0["tries"]), "accepted_dt": r["dts"],
            "e2e": {"value": tot_iter_e2e / (r["ms_e2e"] * 1e-3), "unit": "node-iterations/s",
                    "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "ms_per_step": r["ms_e2e"] / args.steps, "same_steps_as_value": r["same_steps"], "sweeps": int(sweeps_e2e),
                    "host_ms_per_step": {"forcing_upload": r["host_ms"][0], "compute_step": r["host_ms"][1], "result_download_exposed": r["host_ms"][2]},
                    "host_ms_note": "computeStep returns with its accept pass (0.6 ms) still enqueued: the next host-blocking call, the forcing upload, waits for it",
                    "result_download": "sf3d_ext_get_layer_rasters_async into two page-locked buffers: the copy of step k overlaps the kernels of step k + 1 "
                                       "(second CUDA stream); the host waits for it and reads the maps before the next download is issued, the last one "
                                       "inside the timed region",
                    "sim_hours_per_wall_s": r["sim_e2e"] / 3600.0 / (r["ms_e2e"] * 1e-3)},
            "gpu_launches": int(c1["kernel_launches"] - c0["kernel_launches"]),
            "roofline": {"kernel": "kern_jacobi" if world == 1 else "kern_jacobi_multi (sweep + halo stores + residual all-reduce)",
                         "bound": "hbm", "achieved": jac_gbs, "peak": peak, "unit": "GB/s",
                         "frac": (jac_gbs / peak) if jac_gbs else None, "traffic": traffic, "peak_source": peak_src,
                         "bytes_per_launch": bytes_sweep, "avg_launch_ms": jac["ms"] / max(sweeps, 1),
                         "launches": jac["launches"], "executed_sweeps": int(sweeps),
                         "frac_of_nominal_8000": (jac_gbs / 8000.0) if jac_gbs else None,
                         "bytes_representation": bytes_repr,
                         "frac_representation": (bytes_repr * sweeps / jac_s / 1e9 / peak) if jac["ms"] > 0 else None,
                         "frac_traffic": (traffic / (jac["ms"] / max(sweeps, 1) * 1e-3) / 1e9 / peak) if (traffic and jac["ms"] > 0) else None,
                         "note": "achieved / frac count the ALGORITHMIC bytes of SURVEY 8d (12 B per stored entry + 32 B per row); the kernel does "
                                 "not read the 4 B column indices (pattern-compressed: 2 B per row), so frac can exceed 1. frac_representation "
                                 "counts the bytes this representation must move (8 B per entry + 34 B per row); frac_traffic = measured DRAM "
                                 "bytes of one launch (ncu, profiles/jacobi_traffic.json) / time / peak"},
            "roofline_assembly": {"kernel": "kern_node_phase + kern_assemble", "bound": "fp64 issue (HBM reported)",
                                  "achieved": asm_gbs, "peak": peak, "unit": "GB/s", "frac": (asm_gbs / peak) if asm_gbs else None,
                                  "bytes_per_approximation": bytes_asm, "avg_ms_per_approximation": asm_ms / max(approx, 1)},
            "kernel_ms": {k: round(v["ms"], 3) for k, v in ktimes.items()},
            "kernel_share": {k: round(v["ms"] / max(r["ms_profiled"], 1e-9), 4) for k, v in ktimes.items()},
            "kernel_times_from": ("a separate replay of the same accepted steps with a CUDA event pair around every launch (%.3f ms per step with "
                                  "the events, %.3f without: the value region runs without them)" % (r["ms_profiled"] / args.steps, ms / args.steps))
                                 if r["replay"] else "CUDA event pairs around every launch inside the value region",
            "clocks": r["clocks"],
        }
        if args.heat:
            line["roofline_heat"] = heat_roofline(ktimes, c0, c1, N, links, peak)
        if parity is not None:
            line["parity_check"] = parity
        if c4 is not None:
            cN, cl = c4["N"], c4["c1"]["links"]
            cs = c4["sweeps"]
            cj = c4["ktimes"]["jacobi"]
            line["c4"] = {
                "workload": f"C4 slab: {C4_SLAB['rows']}x{C4_SLAB['cols']} DEM per GPU x (1+{C4_SLAB['soil_layers']}) layers, lower third of the layers saturated, "
                            f"free drainage, {RAIN_MM_H:g} mm/h; {world} slab(s) = {C4_SLAB['rows'] * world}x{C4_SLAB['cols']} catchment"
                            + (" = BASELINE configs[3]" if world == 8 else ""),
                "value": c4["owned_global"] * float(cs) / (c4["ms"] * 1e-3), "unit": "node-iterations/s", "steps": args.c4_steps, "warmup": 3,
                "ms_per_step": c4["ms"] / args.c4_steps, "nodes_per_gpu": cN, "sweeps": int(cs),
                "approximations": int(c4["c1"]["approximations"] - c4["c0"]["approximations"]),
                "sim_hours_per_wall_s": c4["sim"] / 3600.0 / (c4["ms"] * 1e-3),
                "sweep_ms": cj["ms"] / max(cs, 1), "sweep_frac_of_peak": ((12.0 * cl + 32.0 * cN) * cs / (cj["ms"] * 1e-3) / 1e9 / peak) if cj["ms"] > 0 else None,
                "kernel_ms": {k: round(v["ms"], 3) for k, v in c4["ktimes"].items() if v["ms"] > 0},
                "clocks": c4["clocks"],
            }
            if parity_c4 is not None:
                line["c4"]["parity_check"] = parity_c4
        if world == 1 and not args.no_cpu_baseline and not args.heat:
            try:
                b = cpu_run(dict(rows=args.rows, cols=args.cols, soil_layers=args.soil_layers, saturated_bottom=args.saturated_bottom),
                            steps=args.steps, warmup=warmup, budget_s=25.0)
                line["cpu_baseline"] = {k: b[k] for k in ("value", "unit", "cores", "kind", "sample")}
                line["cpu_baseline"]["sim_hours_per_wall_s"] = b["sim_hours_per_wall_s"]
                line["cpu_baseline"]["same_accepted_dt_as_gpu"] = b["accepted_dt"] == r["dts"][: len(b["accepted_dt"])]
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "error": str(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def heat_roofline(ktimes, c0, c1, N, links, peak):
    """fractions of the measured HBM peak of the heat kernels, by the algorithmic bytes of SURVEY 8d: heat sweep
    12 B per stored entry + 24 B per row, heat assembly ~200 B per row + 12 B per link + 8 B per entry"""
    hs = int(c1["heat_sweeps"] - c0["heat_sweeps"])
    hsteps = max(1, ktimes["heat_assemble"]["launches"])
    out = {}
    if ktimes["heat_jacobi"]["ms"] > 0 and hs:
        b = 12.0 * links + 24.0 * N
        out["heat_jacobi"] = {"ms_per_sweep": ktimes["heat_jacobi"]["ms"] / hs, "bytes": b,
                              "frac": b * hs / (ktimes["heat_jacobi"]["ms"] * 1e-3) / 1e9 / peak}
    if ktimes["heat_assemble"]["ms"] > 0:
        b = 200.0 * N + 12.0 * links + 8.0 * links
        out["heat_assemble"] = {"ms_per_launch": ktimes["heat_assemble"]["ms"] / hsteps, "bytes": b,
                                "frac": b * hsteps / (ktimes["heat_assemble"]["ms"] * 1e-3) / 1e9 / peak}
    for k in ("heat_coeffs", "heat_flux_snapshot", "heat_boundary", "heat_post", "heat_accept"):
        if ktimes[k]["launches"]:
            out[k] = {"ms_per_launch": ktimes[k]["ms"] / ktimes[k]["launches"], "launches": ktimes[k]["launches"]}
    return out


if __name__ == "__main__":
    main()
