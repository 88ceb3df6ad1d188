"""Run under torchrun (one rank per GPU): the row-slab product against the oracle on the WHOLE catchment.  Every
rank runs the CPU oracle on the full (small) catchment and checks its owned nodes.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29611 tests/mgpu_slab_check.py [--heat] [--timeout-test]

SF3D_SHARE_DEVICE=1: every rank uses cuda:0 (gloo process group, no NCCL communicator: the halo and the all-reduces
run over CUDA-IPC peer memory of the same device).  That is how the multi-rank path is exercised on a one-GPU box.
`slab_parity` is also what bench.py runs before its timed region when WORLD_SIZE > 1 ("parity_check")."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def slab_parity(gpu, rank: int, world: int, *, heat: bool = False, nccl: bool = True, threads: int = 1, c4: bool = False,
                save_all: bool = False) -> dict:
    """48 x 40 x (1+5) storm (water), 24 x 16 x (1+4) coupled heat, or (c4) the C4 recipe at small size -- 32 x 24 x (1+20)
    with the lower third of the layers saturated and free drainage --, split into `world` row slabs, against the
    reference (oracle/_ref when it travelled with the snapshot, else the C restatement) run on the whole catchment
    by every rank.  Returns the comparison; raises nothing (ok False + reason instead)."""
    from criteria3d_b200 import BoundaryType, Field, SoilFluxes3D
    from criteria3d_b200.mgpu import setup_slab
    from criteria3d_b200.synth import Catchment, run_hours, set_heat_forcing, setup
    from oracle import checker_path

    R, C, L = (24, 16, 4) if heat else ((32, 24, 20) if c4 else (48, 40, 5))
    hours, max_steps = ([0.0, 10.0], 10) if heat else (([40.0], 25) if c4 else ([20.0, 40.0], 50))
    cat_kw = dict(saturated_bottom=True) if c4 else {}
    # save_all: heat flux save mode All (every flux type kept per link), which also runs the water-flux snapshot pass
    hf_mode = 2 if (heat and save_all) else None
    slab, lc = setup_slab(gpu, R, C, L, rank, world, heat=heat, require_direct=not nccl, heat_flux_mode=hf_mode, **cat_kw)
    launches0 = gpu.counters()["kernel_launches"]

    def run(sf, cat):
        dts = []
        for h, mm in enumerate(hours):
            if heat:
                set_heat_forcing(sf, cat, 10 + h)
            dts += run_hours(sf, cat, [mm], max_steps=max_steps)
        return dts
    dts = run(gpu, lc)
    launches = int(gpu.counters()["kernel_launches"] - launches0)
    chk = SoilFluxes3D(checker_path())
    cat = Catchment(R, C, L, heat=heat, **cat_kw)
    setup(chk, cat, threads=threads, heat_flux_mode=hf_mode)
    dts_ref = run(chk, cat)

    out = {"world": world, "grid": f"{R}x{C}x(1+{L})" + (" coupled heat" if heat else "") + (", save mode All" if hf_mode else "") + (" saturated lower third (C4 recipe)" if c4 else ""), "checker": chk.backend,
           "halo": getattr(gpu, "halo_mode", "?"), "steps": len(dts), "dt_sequence_equal": dts == dts_ref, "launches": launches, "ok": True, "why": []}
    if dts != dts_ref:
        out["ok"] = False
        out["why"].append("accepted time steps differ")
    own, l2g = slab.owned_mask(), slab.local_to_global()
    fields = [(Field.TOTAL_POTENTIAL, 1e-6, "max_dH_rel"), (Field.WATER_CONTENT, 1e-7, "max_dtheta"), (Field.DEGREE_OF_SATURATION, 1e-6, "max_dSe")]
    if heat:
        fields.append((Field.TEMPERATURE, 1e-6, "max_dT_rel"))
    for f, tol, key in fields:
        a = gpu.get_field(f, 0, lc.n_nodes)[own]
        b = chk.get_field(f, 0, cat.n_nodes)[l2g[own]]
        if f == Field.TEMPERATURE:                      # surface nodes carry the TopographyError sentinel on both sides
            keep = l2g[own] >= cat.n_surface
            a, b = a[keep], b[keep]
        err = float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) if a.size else 0.0
        out[key] = err
        if not err <= tol:
            out["ok"] = False
            out["why"].append(f"{f.name} err {err:.3e} > {tol}")
    if hf_mode:
        # the water-flux snapshot of the heat step (flux types 5..8 of types.h:199, float-rounded), Down direction, on a
        # sample of owned soil nodes: computed by a pass of its own that only runs in this save mode / with advection
        owned_soil = np.flatnonzero(own & (np.arange(lc.n_nodes) >= lc.n_surface))
        pick = owned_soil[:: max(1, owned_soil.size // 40)]
        a = np.array([[gpu.getNodeHeatMaxFlux(int(i), 2, t) for t in range(5, 9)] for i in pick])
        b = np.array([[chk.getNodeHeatMaxFlux(int(l2g[i]), 2, t) for t in range(5, 9)] for i in pick])
        scale = np.maximum(np.abs(b), 1e-12 + 1e-6 * np.max(np.abs(b)))
        err = float(np.max(np.abs(a - b) / scale))
        out["max_dWaterFluxSnapshot_rel"] = err
        if not (err <= 1e-4 and np.any(b != 0)):          # float-rounded values of differences of nearly equal heads
            out["ok"] = False
            out["why"].append(f"water flux snapshot err {err:.3e}")
    tw, tw_ref = gpu.getTotalWaterContent(), chk.getTotalWaterContent()
    out["total_water_rel"] = abs(tw - tw_ref) / abs(tw_ref)
    if not out["total_water_rel"] <= 1e-9:
        out["ok"] = False
        out["why"].append("total water")
    for bt in (BoundaryType.Runoff, BoundaryType.FreeDrainage, BoundaryType.FreeLateralDrainage):
        a, b = gpu.getTotalBoundaryWaterFlow(int(bt)), chk.getTotalBoundaryWaterFlow(int(bt))
        if not abs(a - b) <= 1e-6 * abs(b) + 1e-12:
            out["ok"] = False
            out["why"].append(f"boundary total {bt.name}: {a} vs {b}")
    cg, cr = gpu.counters(), chk.counters()
    out["sweeps"] = [int(cg["sweeps"]), int(cr["sweeps"])]
    out["approximations"] = [int(cg["approximations"]), int(cr["approximations"])]
    if cg["approximations"] != cr["approximations"]:
        out["ok"] = False
        out["why"].append("approximation count")
    return out


def reduce_over_ranks(out: dict) -> dict:
    """worst case over the ranks (every rank checked its own slab).  Every rank must have launched the same kernels:
    the ranks take the same decisions (same transport, same sweeps), so unequal counts mean a mixed-form run."""
    import torch.distributed as dist
    alls = [None] * dist.get_world_size()
    dist.all_gather_object(alls, out)
    merged = dict(alls[0])
    merged["ok"] = all(o["ok"] for o in alls)
    merged["dt_sequence_equal"] = all(o["dt_sequence_equal"] for o in alls)
    merged["why"] = sorted({w for o in alls for w in o["why"]})
    launches = [o["launches"] for o in alls]
    if len(set(launches)) != 1:
        merged["ok"] = False
        merged["why"].append(f"kernel launches differ between ranks: {launches}")
    for k in ("max_dH_rel", "max_dtheta", "max_dSe", "max_dT_rel", "total_water_rel"):
        if k in merged:
            merged[k] = max(o[k] for o in alls)
    return merged


def timeout_check(gpu, rank: int, world: int) -> dict:
    """A rank that stops answering must surface as an ERROR on its peers, never as different physics: rank 1 does
    not call computeStep; rank 0's computeStep has to come back within the mailbox time-out with a negative
    sentinel, sf3d_ext_last_error() == SolverError, and keep failing (sticky) instead of accepting a garbage step."""
    import time
    import torch.distributed as dist
    from criteria3d_b200 import Field, SF3Derror
    from criteria3d_b200.mgpu import setup_slab
    slab, lc = setup_slab(gpu, 48, 40, 5, rank, world, require_direct=True)
    sink = np.zeros(lc.n_nodes)
    sink[: lc.n_surface] = lc.rain_sink_source(20.0)
    gpu.set_field(Field.WATER_SINK_SOURCE, 0, sink)
    out = {"ok": True}
    if rank == 0:
        t0 = time.perf_counter()
        dt = gpu.computeStep(3600.0)
        out.update({"returned": dt, "seconds": time.perf_counter() - t0, "last_error": int(gpu.last_error())})
        dt2 = gpu.computeStep(3600.0)
        out["second_call"] = dt2
        out["ok"] = dt < 0 and out["last_error"] == int(SF3Derror.SolverError) and dt2 < 0 and out["seconds"] < 30.0
    dist.barrier()
    return out


def main():
    import torch
    import torch.distributed as dist
    from criteria3d_b200 import load_product
    from criteria3d_b200.mgpu import wire_ranks
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    share = os.environ.get("SF3D_SHARE_DEVICE", "0") == "1"
    dev_index = 0 if share else local
    torch.cuda.set_device(dev_index)
    if share:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev_index))
    gpu = load_product()
    assert gpu.set_device(dev_index) == 0
    wire_ranks(gpu, rank, world, nccl=not share)
    if "--timeout-test" in sys.argv:
        out = timeout_check(gpu, rank, world)
        if rank == 0:
            print(f"[mgpu_slab_check] timeout {'ok' if out['ok'] else 'FAILED'}: {out}", flush=True)
        dist.barrier()
        dist.destroy_process_group()
        sys.exit(0 if out["ok"] else 1)
    heat = "--heat" in sys.argv
    out = reduce_over_ranks(slab_parity(gpu, rank, world, heat=heat, nccl=not share, c4="--c4" in sys.argv, save_all="--save-all" in sys.argv))
    dist.barrier()
    if rank == 0:
        print(f"[mgpu_slab_check] {'ok' if out['ok'] else 'FAILED'}: {out}", flush=True)
    gpu.comm_finalize()
    dist.destroy_process_group()
    sys.exit(0 if out["ok"] else 1)


if __name__ == "__main__":
    main()
