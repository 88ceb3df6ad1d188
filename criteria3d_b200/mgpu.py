"""Harness plumbing for the row-slab multi-GPU path: one process per GPU (torchrun), the NCCL unique id and the
CUDA IPC handles exchanged through torch.distributed (any backend: object collectives), slab catchment set up
through the ordinary C ABI."""
from __future__ import annotations

import os

import torch
import torch.distributed as dist

from .capi import SoilFluxes3D
from .partition import Slab, make_slab, slab_catchment
from .synth import Catchment, _ok, setup


def wire_ranks(sf: SoilFluxes3D, rank: int, world: int, device: torch.device | None = None, *, nccl: bool = True) -> None:
    """Create the library's communicator over the already initialised torch process group.
    nccl=False: peer memory only (no NCCL communicator), e.g. when the ranks share one device."""
    if not nccl:
        _ok(sf.comm_init(rank, world, None), "sf3d_ext_comm_init")
        return
    box = [sf.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    _ok(sf.comm_init(rank, world, box[0]), "sf3d_ext_comm_init")


def setup_slab(sf: SoilFluxes3D, rows: int, cols: int, n_soil_layers: int, rank: int, world: int,
               numerics=None, require_direct: bool = False, heat_flux_mode: int | None = None, **cat_kw) -> tuple[Slab, Catchment]:
    """initialize3DModel's sequence on this rank's slab (owned rows + ghost rows), then the halo lists.
    The balance is initialised after the ghosts are known so that storage counts owned nodes only."""
    slab = make_slab(rows, cols, n_soil_layers, world, rank)
    cat = slab_catchment(slab, **cat_kw)
    setup(sf, cat, numerics=numerics, heat_flux_mode=heat_flux_mode, balance=(world == 1))
    if world > 1:
        peers, send, recv = slab.halo()
        _ok(sf.set_halo(peers, send, recv, slab.n_global), "sf3d_ext_set_halo")
        if require_direct or os.environ.get("SF3D_DIRECT_HALO", "1") != "0":
            ok = 1
            try:
                wire_direct_halo(sf, slab, peers)
            except Exception as e:  # noqa: BLE001  (e.g. no peer access between two devices)
                if require_direct:
                    raise
                print(f"[sf3d] rank {rank}: direct peer-memory wiring failed ({e}); falling back to NCCL", flush=True)
                ok = 0
            # the ranks must agree: one failure puts everybody back on the NCCL halo / all-reduce
            flags = [None] * world
            dist.all_gather_object(flags, ok)
            if min(flags) == 0:
                _ok(sf.set_halo(peers, send, recv, slab.n_global), "sf3d_ext_set_halo")      # drops every IPC mapping
            sf.halo_mode = "peer-memory" if min(flags) else "nccl"
        else:
            sf.halo_mode = "nccl"
        _ok(sf.initializeBalance(), "initializeBalance")
    return slab, cat


def wire_direct_halo(sf: SoilFluxes3D, slab: Slab, peers) -> None:
    """Exchange the CUDA IPC handles of every rank's solution buffers and mailbox and tell the library where each
    send entry lives in the neighbour's numbering (= the neighbour's recv list towards this rank)."""
    blob = sf.ipc_export() + sf.mailbox_export()
    blobs = [None] * slab.world
    dist.all_gather_object(blobs, blob)
    for p in peers:
        other = make_slab(slab.rows, slab.cols, slab.layers - 1, slab.world, p)
        o_peers, _o_send, o_recv = other.halo()
        remote = o_recv[o_peers.index(slab.rank)]
        _ok(sf.ipc_import(p, blobs[p][:128], remote), "sf3d_ext_ipc_import")
    for p in range(slab.world):
        if p != slab.rank:
            _ok(sf.mailbox_import(p, blobs[p][128:192]), "sf3d_ext_mailbox_import")
