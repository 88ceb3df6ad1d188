// sf3d_backend.h -- the device-side services the host engine uses: memory, copies and one
// launcher per kernel.  Implemented in sf3d_kernels.cu (CUDA, sm_100a).  There is exactly one
// implementation; if CUDA is unavailable every entry point throws (no CPU fallback).
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "sf3d_view.h"
#include "sf3d.h"

namespace sf3d {

struct DeviceError { int code; const char *what; const char *where; };

// ---- memory / transfers (all on the library's stream) ------------------------------------
void   dev_select(int device);          // cudaSetDevice + stream creation (idempotent)
int    dev_current();
void  *dev_alloc(size_t bytes);          // cudaMalloc + zero fill (reference uses calloc)
void   dev_free(void *p);
void   dev_zero(void *p, size_t bytes);
void   dev_fill_f64(double *p, size_t n, double value);
void   dev_copy(void *dst, const void *src, size_t bytes);      // device to device
void   h2d(void *dst, const void *src, size_t bytes);
void   d2h(void *dst, const void *src, size_t bytes);
// overlapped device-to-host copy (second stream): the copy starts after everything enqueued on the library's stream so far and
// runs beside later work; `slot` (0 / 1) names the staging buffer it reads, so that overlap_acquire(slot) can make the library's
// stream wait for that copy before the buffer is written again
void   overlap_acquire(int slot);
void   d2h_overlapped(void *dst, const void *src, size_t bytes, int slot);
void   overlap_sync();
void  *pinned_alloc(size_t bytes);
void   pinned_free(void *p);
void   dev_sync();
uint64_t launches();                     // kernels launched by this library so far
void  *dev_stream();                     // cudaStream_t of the library (for event timing)
void   prof_enable(bool on);             // CUDA-event timing of every launch, per kernel kind
void   prof_get(double ms[SF3D_K_COUNT], uint64_t n[SF3D_K_COUNT]);
uint64_t k_count_links(const SF3DView &v);

// ---- row-slab ranks (NCCL resolved at run time; see sf3d_kernels.cu) ------------------------
void comm_unique_id(unsigned char out[128]);
void comm_init(int rank, int world, const unsigned char id[128]);
void comm_finalize();
int  comm_world();
int  comm_rank();
void comm_clear_halo();
void comm_add_halo_peer(int peer, uint32_t nSend, const uint32_t *sendIdx, uint32_t nRecv, const uint32_t *recvIdx);
void comm_mailbox_export(unsigned char out[64]);
void comm_mailbox_import(int peer, const unsigned char handle[64]);
void comm_mark_boundary(uint16_t *pid);     // boundary rows of the peer-transport sweep (after every pattern build)
void comm_ipc_export(double *x0, double *x1, unsigned char out[128]);
void comm_ipc_import(int peer, const unsigned char handles[128], uint32_t n, const uint32_t *remoteIdx);

// ---- kernels -----------------------------------------------------------------------------
int  reduce_blocks(uint32_t n);          // grid size used by all reducing kernels for n rows
int  wide_blocks(uint32_t n);            // grid size of the node-phase / assembly kernels
void k_link_geometry(const SF3DView &v, int *surfaceOrderOk);
void k_heat_geometry(const SF3DView &v);       // static per-node pressure and per-link 3-D distance
bool k_build_patterns(const SF3DView &v, uint16_t *pid, int32_t *table, uint32_t *hotPid, int32_t hotOff[SF3D_NLINK]);   // pattern-compressed column indices
size_t pattern_table_bytes();
bool k_jacobi_persistent_ok(const SF3DView &v);     // small graphs: all sweeps of a solve in one cooperative launch
void k_jacobi_persistent(const SF3DView &v, double *xa, double *xb, int maxIter, double tol);
void k_begin_try(const SF3DView &v);
void k_restore_old(const SF3DView &v);
void k_node_phase(const SF3DView &v, double dt, int withCapacity);
void k_assemble(const SF3DView &v, double dt, int approx, double dtMin);
void k_jacobi(const SF3DView &v, const double *xin, double *xout, int maxIter, double tol);
void k_post(const SF3DView &v, const double *x, double dt, int mode);
bool k_post_can_follow_solve(const SF3DView &v);   // post pass enqueued behind the sweeps: one control read per approximation
void k_post_follow_solve(const SF3DView &v, int start, double dt, double dtMin);
void k_accept(const SF3DView &v, double dt, bool prepareNextTry);
void k_restore_best(const SF3DView &v);
void k_total_boundary_flow(const SF3DView &v, uint32_t boundaryType);
// coupled heat
void k_update_conductance(const SF3DView &v);
void k_save_water_fluxes(const SF3DView &v, double dtHeat, double dtWater);
void k_reset_water_fluxes(const SF3DView &v);
void k_boundary_heat(const SF3DView &v, double maxTimeStep);
void k_heat_begin(const SF3DView &v, double dtHeat, double dtWater, bool coeffsAreCurrent);   // coeffsAreCurrent: the per-node
                                    // coefficients stored by k_save_water_fluxes were computed with the same (dtHeat, T): not recomputed
void k_heat_assemble(const SF3DView &v, double dtHeat, double dtWater);
void k_heat_jacobi(const SF3DView &v, const double *xin, double *xout, int maxIter, double tol);
void k_heat_post(const SF3DView &v, const double *x, double dtHeat, double dtWater, int mode);
void k_heat_accept(const SF3DView &v, double dtHeat, double dtWater);
void k_heat_copy_T(const SF3DView &v, int mode);
void read_ctrl(const SF3DView &v, Ctrl *out);     // async copy to pinned + stream sync
void write_ctrl(const SF3DView &v, const Ctrl *in);

// bulk field access (device kernels; first/count in nodes)
void k_set_potential(const SF3DView &v, uint32_t first, uint32_t count, const double *src, int isTotal);
void k_get_field(const SF3DView &v, int field, uint32_t first, uint32_t count, double *dst);

// device-side DEM -> graph builder (sf3d_ext_build_grid)
struct GridDev {
    uint32_t rows, cols, layers, nValid;
    double cell, xll, yll;
    const float *dem, *slope;
    const int32_t *rank;
    const uint8_t *outlet, *boundaryL1;
    const uint16_t *soilId, *surfaceId;
    const double *pond;
    const double *layerDepth, *layerThickness;
    const uint16_t *layerTab;       // [layers * nSoilIds]: soil-table row of (soil id, layer horizon)
    uint32_t nSoilIds;
    int freeRunoff, freeLateral, freeBottom;
    int computeWater, computeHeat, heatSurfaceL1;
};
void k_build_grid(const SF3DView &v, const GridDev &g);

// the raster side of a graph built by sf3d_ext_build_grid: node(layer, cell) = layer * nValid + rank[cell]
struct RasterDev {
    uint32_t rows, cols, layers, nValid;
    double cell;
    const int32_t *rank;            // rows*cols, -1 outside the catchment
};
struct ForcingDev {
    const float *precipitation; float precipitationNodata;
    uint32_t nSinkLayers; const float *layerSink; float sinkNodata;
    int accumulate;
};

void k_forcing_rasters(const SF3DView &v, const RasterDev &g, const ForcingDev &f);
void k_layer_raster(const SF3DView &v, const RasterDev &g, int field, uint32_t layer, float nodata, float *dst);

}  // namespace sf3d
