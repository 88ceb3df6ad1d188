/*
 * sf3d.h -- C ABI of the B200-native soilFluxes3D time step.
 *
 * One entry point per free function of the reference plugin API
 * (agrolib/soilFluxes3D/soilFluxes3D.h:9-104, namespace soilFluxes3D::v2).  The C++
 * drop-in shim (include/soilFluxes3D.h + criteria3d_b200/csrc/sf3d_shim.cpp) forwards
 * every reference call to the function of the same row below; the reference-side
 * binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions (same as the reference, soilFluxes3D.cpp):
 *   - single global instance, not thread safe, library owns all memory;
 *   - setters return an SF3Derror_t code as uint8_t (types.h:39-40):
 *       0 Ok, 1 IndexError, 2 MemoryError, 3 TopographyError, 4 BoundaryError,
 *       5 MissingDataError, 6 ParameterError, 7 SolverError, 8 FileError;
 *   - getters return the value or a sentinel double (types.h:42-64):
 *       -1111 index, -2222 memory, -3333 topography, -4444 boundary,
 *       -9999 missing data, -7777 parameter;
 *   - enums cross the boundary as their underlying uint8_t values:
 *       boundaryType_t (types.h:98-99)  0 NoBoundary 1 Runoff 2 FreeDrainage
 *           3 FreeLateralDrainage 4 PrescribedTotalWaterPotential 5 Urban 6 Road
 *           7 Culvert 8 HeatSurface 9 SoluteFlux
 *       linkType_t (types.h:101)        0 NoLink 1 Up 2 Down 3 Lateral
 *       WRCModel (types.h:135)          0 VanGenuchten 1 ModifiedVanGenuchten 2 Campbell
 *       meanType_t (types.h:36)         0 Arithmetic 1 Geometric 2 Logarithmic
 *       heatFluxSaveMode_t (types.h:186) 0 None 1 Total 2 All
 *       fluxTypes_t (types.h:199)       0 HeatTotal .. 8 WaterVaporThermal
 *
 * The same header is implemented by three libraries so that one harness drives all:
 *   criteria3d_b200/libsf3d_b200.so   the product (CUDA, sm_100a; no CPU fallback)
 *   oracle/libsf3d_oracle.so          the CPU restatement (test infrastructure only)
 *   oracle/_ref/libsf3d_ref.so        the unmodified reference sources behind this ABI
 */
#ifndef SF3D_H
#define SF3D_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SF3D_OK                 0
#define SF3D_INDEX_ERROR        1
#define SF3D_MEMORY_ERROR       2
#define SF3D_TOPOGRAPHY_ERROR   3
#define SF3D_BOUNDARY_ERROR     4
#define SF3D_MISSING_DATA_ERROR 5
#define SF3D_PARAMETER_ERROR    6
#define SF3D_SOLVER_ERROR       7
#define SF3D_FILE_ERROR         8

#define SF3D_MAX_LATERAL_LINK 8   /* types.h:24 */
#define SF3D_MAX_TOTAL_LINK   10  /* types.h:25 */

/* ---- initialisation and memory management (soilFluxes3D.h:9-21) ---------------- */
uint8_t  sf3d_initialize(uint32_t nrNodes, uint32_t nrSurfaceNodes, uint8_t nrLateralLinks,
                         int isComputeWater, int isComputeHeat, int isComputeSolutes,
                         uint8_t heatFluxSaveMode);                /* initializeSF3D      :10 */
uint8_t  sf3d_initialize_balance(void);                            /* initializeBalance   :14 */
uint8_t  sf3d_clean(void);                                         /* cleanSF3D           :17 */
uint8_t  sf3d_initialize_heat_flag(uint8_t saveModeHeat, int isComputeAdvectiveFlux,
                                   int isComputeLatentHeat);       /* initializeHeatFlag  :20 */
uint32_t sf3d_set_threads_number(uint32_t nrThreads);              /* setThreadsNumber    :22 */
void     sf3d_set_use_lineal(int value);                           /* setUseLineal        :23 */
void     sf3d_set_lineal_method(int value);                        /* setLinealMethod     :24 */

/* ---- soil / surface tables (soilFluxes3D.h:27-30) ------------------------------- */
uint8_t sf3d_set_soil_properties(uint16_t nrSoil, uint8_t nrHorizon, double VG_alpha, double VG_n,
                                 double VG_m, double VG_he, double thetaR, double thetaS, double kSat,
                                 double MualemL, double organicMatter, double clay);
uint8_t sf3d_set_surface_properties(uint16_t surfaceIndex, double roughness);

/* ---- core parameters (soilFluxes3D.h:33-34) ------------------------------------- */
uint8_t sf3d_set_numerical_parameters(double minDeltaT, double maxDeltaT, uint16_t maxIterationNumber,
                                      uint16_t maxApproximationsNumber, uint8_t residualToleranceExponent,
                                      uint8_t MBRThresholdExponent);
uint8_t sf3d_set_hydraulic_properties(uint8_t waterRetentionCurve, uint8_t conductivityMeanType,
                                      float conductivityHorizVertRatio);

/* ---- topology (soilFluxes3D.h:37-40) -------------------------------------------- */
uint8_t sf3d_set_culvert(uint32_t nodeIndex, double roughness, double slope, double width, double height);
uint8_t sf3d_set_node(uint32_t index, double x, double y, double z, double volume_or_area, int isSurface,
                      uint8_t boundaryType, double slope, double boundaryArea);
uint8_t sf3d_set_node_link(uint32_t nodeIndex, uint32_t linkIndex, uint8_t direction, double interfaceArea);
uint8_t sf3d_set_node_boundary(uint32_t nodeIndex, uint8_t boundaryType, double slope, double boundaryArea);

/* ---- soil data (soilFluxes3D.h:43-44) ------------------------------------------- */
uint8_t sf3d_set_node_soil(uint32_t nodeIndex, uint16_t soilIndex, uint16_t horizonIndex);
uint8_t sf3d_set_node_surface(uint32_t nodeIndex, uint16_t surfaceIndex);

/* ---- water setters (soilFluxes3D.h:47-53) --------------------------------------- */
uint8_t sf3d_set_node_pond(uint32_t nodeIndex, double pond);
uint8_t sf3d_set_node_water_content(uint32_t nodeIndex, double waterContent);
uint8_t sf3d_set_node_degree_of_saturation(uint32_t nodeIndex, double degreeOfSaturation);
uint8_t sf3d_set_node_matric_potential(uint32_t nodeIndex, double matricPotential);
uint8_t sf3d_set_node_total_potential(uint32_t nodeIndex, double totalPotential);
uint8_t sf3d_set_node_water_sink_source(uint32_t nodeIndex, double waterSinkSource);
uint8_t sf3d_set_node_prescribed_total_potential(uint32_t nodeIndex, double prescribedTotalPotential);

/* ---- water getters (soilFluxes3D.h:56-74) --------------------------------------- */
double sf3d_get_node_water_content(uint32_t nodeIndex);
double sf3d_get_node_maximum_water_content(uint32_t nodeIndex);
double sf3d_get_node_minimum_water_content(uint32_t nodeIndex);
double sf3d_get_node_available_water_content(uint32_t nodeIndex);
double sf3d_get_node_water_deficit(uint32_t nodeIndex, double fieldCapacity);
double sf3d_get_node_degree_of_saturation(uint32_t nodeIndex);
double sf3d_get_node_water_conductivity(uint32_t nodeIndex);
double sf3d_get_node_matric_potential(uint32_t nodeIndex);
double sf3d_get_node_total_potential(uint32_t nodeIndex);
double sf3d_get_node_pond(uint32_t nodeIndex);
double sf3d_get_node_max_water_flow(uint32_t nodeIndex, uint8_t linkDirection);
double sf3d_get_node_sum_lateral_water_flow(uint32_t nodeIndex);
double sf3d_get_node_sum_lateral_water_flow_in(uint32_t nodeIndex);
double sf3d_get_node_sum_lateral_water_flow_out(uint32_t nodeIndex);
double sf3d_get_node_boundary_water_flow(uint32_t nodeIndex);
double sf3d_get_total_boundary_water_flow(uint8_t boundaryType);
double sf3d_get_total_water_content(void);
double sf3d_get_water_storage(void);
double sf3d_get_water_mbr(void);

/* ---- heat setters (soilFluxes3D.h:77-86) ---------------------------------------- */
uint8_t sf3d_set_node_heat_sink_source(uint32_t nodeIndex, double heatSinkSource);
uint8_t sf3d_set_node_temperature(uint32_t nodeIndex, double temperature);
uint8_t sf3d_set_node_boundary_fixed_temperature(uint32_t nodeIndex, double fixedTemperature, double depth);
uint8_t sf3d_set_node_boundary_height_wind(uint32_t nodeIndex, double heightWind);
uint8_t sf3d_set_node_boundary_height_temperature(uint32_t nodeIndex, double heightTemperature);
uint8_t sf3d_set_node_boundary_net_irradiance(uint32_t nodeIndex, double netIrradiance);
uint8_t sf3d_set_node_boundary_temperature(uint32_t nodeIndex, double temperature);
uint8_t sf3d_set_node_boundary_relative_humidity(uint32_t nodeIndex, double relativeHumidity);
uint8_t sf3d_set_node_boundary_roughness(uint32_t nodeIndex, double roughness);
uint8_t sf3d_set_node_boundary_wind_speed(uint32_t nodeIndex, double windSpeed);

/* ---- heat getters (soilFluxes3D.h:89-101) --------------------------------------- */
double sf3d_get_node_temperature(uint32_t nodeIndex);
double sf3d_get_node_heat_conductivity(uint32_t nodeIndex);
double sf3d_get_node_vapor(uint32_t nodeIndex);
double sf3d_get_node_heat_storage(uint32_t nodeIndex, double h);
double sf3d_get_node_heat_max_flux(uint32_t nodeIndex, uint8_t linkDirection, uint8_t fluxType);
double sf3d_get_node_boundary_advective_flux(uint32_t nodeIndex);
double sf3d_get_node_boundary_latent_flux(uint32_t nodeIndex);
double sf3d_get_node_boundary_radiative_flux(uint32_t nodeIndex);
double sf3d_get_node_boundary_sensible_flux(uint32_t nodeIndex);
double sf3d_get_node_boundary_aerodynamic_conductance(uint32_t nodeIndex);
double sf3d_get_node_boundary_soil_conductance(uint32_t nodeIndex);
double sf3d_get_heat_mbr(void);
double sf3d_get_heat_mbe(void);

/* ---- computation (soilFluxes3D.h:103-104) --------------------------------------- */
void   sf3d_compute_period(double timePeriod);
double sf3d_compute_step(double maxTimeStep);

/* =================================================================================
 * Extensions (not in the reference API).  They exist because the reference is driven by
 * O(10 N) scalar calls (project3D.cpp:941-1103, 2269-2285, 2763-2797), which is the new
 * bottleneck once the step itself runs on a B200.  Every extension is defined as "the
 * same as calling the scalar function for each node of the range", so the reference
 * library can (and in oracle/_ref does) implement it as a plain loop.
 * ================================================================================= */

/* quantities addressable in bulk; GET mirrors the scalar getter, SET the scalar setter */
enum sf3d_field {
    SF3D_F_WATER_CONTENT        = 0,  /* get/set NodeWaterContent            */
    SF3D_F_DEGREE_OF_SATURATION = 1,  /* get/set NodeDegreeOfSaturation      */
    SF3D_F_WATER_CONDUCTIVITY   = 2,  /* getNodeWaterConductivity            */
    SF3D_F_MATRIC_POTENTIAL     = 3,  /* get/set NodeMatricPotential         */
    SF3D_F_TOTAL_POTENTIAL      = 4,  /* get/set NodeTotalPotential          */
    SF3D_F_POND                 = 5,  /* get/set NodePond (surface nodes)    */
    SF3D_F_WATER_SINK_SOURCE    = 6,  /* setNodeWaterSinkSource (set only)   */
    SF3D_F_BOUNDARY_WATER_FLOW  = 7,  /* getNodeBoundaryWaterFlow            */
    SF3D_F_PRESCRIBED_POTENTIAL = 8,  /* setNodePrescribedTotalPotential     */
    SF3D_F_TEMPERATURE          = 9,  /* get/set NodeTemperature             */
    SF3D_F_HEAT_SINK_SOURCE     = 10, /* setNodeHeatSinkSource               */
    SF3D_F_SUM_LATERAL_FLOW     = 11, /* getNodeSumLateralWaterFlow          */
    SF3D_F_MAX_FLOW_UP          = 12, /* getNodeMaxWaterFlow(Up)             */
    SF3D_F_MAX_FLOW_DOWN        = 13, /* getNodeMaxWaterFlow(Down)           */
    SF3D_F_MAX_FLOW_LATERAL     = 14, /* getNodeMaxWaterFlow(Lateral)        */
    SF3D_F_HEAT_CONDUCTIVITY    = 15, /* getNodeHeatConductivity             */
    SF3D_F_BOUNDARY_NET_IRRADIANCE = 16, /* setNodeBoundaryNetIrradiance     */
    SF3D_F_BOUNDARY_TEMPERATURE = 17,    /* setNodeBoundaryTemperature       */
    SF3D_F_BOUNDARY_RELATIVE_HUMIDITY = 18,
    SF3D_F_BOUNDARY_WIND_SPEED  = 19,
    SF3D_F_BOUNDARY_HEIGHT_WIND = 20,        /* setNodeBoundaryHeightWind        */
    SF3D_F_BOUNDARY_HEIGHT_TEMPERATURE = 21, /* setNodeBoundaryHeightTemperature */
    SF3D_F_BOUNDARY_ROUGHNESS   = 22,        /* setNodeBoundaryRoughness         */
    SF3D_F_COUNT
};

/* dst/src are HOST buffers of `count` doubles for nodes [first, first+count).
 * Return: 0 or the first non-zero SF3Derror_t met (get: sentinels are stored as values). */
uint8_t sf3d_ext_get_field(int field, uint32_t first, uint32_t count, double *dst);
uint8_t sf3d_ext_set_field(int field, uint32_t first, uint32_t count, const double *src);

/* integer maps (bit-exact parity surface): link slot table as the reference stores it
 * (slot 0 Up, 1 Down, 2.. Lateral; soilFluxes3D.cpp:644-664).  index = 0xFFFFFFFF... is
 * never produced: an empty slot reports type 0 (NoLink) and index 0 (calloc'ed). */
uint8_t sf3d_ext_get_link_table(uint8_t slot, uint32_t first, uint32_t count,
                                uint8_t *linkType, uint32_t *linkIndex, double *interfaceArea);
uint8_t sf3d_ext_get_node_meta(uint32_t first, uint32_t count, uint8_t *surfaceFlag,
                               uint8_t *boundaryType, uint8_t *numLateralLink);

/* Bulk DEM -> node/link graph builder: the recipe of Project3D::setIndexMaps +
 * setCrit3DTopography + setCrit3DNodeSoil (src/project3D/project3D.cpp:758-818, 941-1103,
 * 1164-1238) for a raster whose valid cells are the same on every layer.
 *   node index  = layer * n_valid + cell_rank[row*cols+col]   (layer-major, row-major)
 *   x = x_ll + (col+0.5)*cell ; y = y_ll + (rows-row-0.5)*cell  (gis getXY convention)
 *   z = (float)(dem - (float)layer_depth[layer])                 (float arithmetic, :966)
 * Must be called after sf3d_initialize(layers*n_valid, n_valid, 8, ...) and after the soil
 * and surface tables are set.  Calls (conceptually) setNode, setNodeLink (Up, Down, 8
 * Lateral in (dr,dc) order (-1,-1)..(1,1)), setNodeSurface + setNodePond | setNodeSoil. */
typedef struct sf3d_grid_desc {
    uint32_t rows, cols, layers;      /* layers includes layer 0 = surface               */
    uint32_t n_valid;                 /* number of valid cells                            */
    double   cell;                    /* [m]                                              */
    double   x_ll, y_ll;              /* lower-left corner                                */
    const float    *dem;              /* rows*cols, [m]                                   */
    const float    *slope_tan;        /* rows*cols, tan(slope) already in float           */
    const int32_t  *cell_rank;        /* rows*cols, -1 = NODATA cell                      */
    const uint8_t  *outlet;           /* rows*cols, 1 = boundaryMap == BOUNDARY_RUNOFF    */
    const uint16_t *soil_id;          /* rows*cols                                        */
    const uint16_t *surface_id;       /* rows*cols                                        */
    const double   *pond;             /* rows*cols, [m]                                   */
    const double   *layer_depth;      /* layers, centre depth [m]                         */
    const double   *layer_thickness;  /* layers, [m] (layer 0: 0)                         */
    const uint16_t *layer_horizon;    /* layers, horizon index used by setNodeSoil        */
    const uint8_t  *boundary_l1;      /* rows*cols or NULL: 5 Urban / 6 Road on layer 1   */
    int free_catchment_runoff, free_lateral_drainage, free_bottom_drainage;
    int heat_surface_layer1;          /* 1: layer-1 nodes get the HeatSurface boundary (setNodeBoundary
                                         after setNode; replaces drainage / urban / road on that layer) */
} sf3d_grid_desc;
uint8_t sf3d_ext_build_grid(const sf3d_grid_desc *desc);

/* Raster-facing forcing and output for a graph built by sf3d_ext_build_grid (SURVEY 8 f3, f4).
 *
 * sf3d_ext_set_forcing_rasters: the hourly forcing assembly of the caller, in the caller's order
 * (bin/CRITERIA3D/criteria3DProject.cpp:2121-2160): sink/source := 0 on every node (:2123-2127), then
 * for every valid cell and every layer l < n_sink_layers with s = layer_sink[l][cell] != nodata, s > 0
 *     sink[node(l, cell)] -= area * (s / 1000.) / 3600.     (assignEvaporation / assignTranspiration,
 *                                                            src/project3D/project3D.cpp:2397-2401, 2436-2440, 2603)
 * then with p = precipitation[cell] != nodata, p > 0
 *     flow = area * (p / 1000.) ; if (flow / 3600. > 0) sink[node(0, cell)] += flow / 3600.
 *                                                           (assignPrecipitation, criteria3DProject.cpp:939-965)
 * and Project3D::setSinkSource (project3D.cpp:2269-2285).  Values are float rasters [mm h-1] as the
 * reference's meteo maps; area = cell * cell.  accumulate != 0 skips the zeroing.
 * Errors: SF3D_MISSING_DATA_ERROR when no grid was built, SF3D_PARAMETER_ERROR on a shape mismatch. */
typedef struct sf3d_forcing_desc {
    uint32_t rows, cols;              /* must equal the built grid                                  */
    const float *precipitation;       /* rows*cols [mm h-1] liquid water reaching the surface, or NULL */
    float precipitation_nodata;
    uint32_t n_sink_layers;           /* layer_sink covers layers 0 .. n_sink_layers-1 (0 = surface) */
    const float *layer_sink;          /* [n_sink_layers][rows*cols] [mm h-1] water removed, or NULL  */
    float sink_nodata;
    int accumulate;
} sf3d_forcing_desc;
uint8_t sf3d_ext_set_forcing_rasters(const sf3d_forcing_desc *desc);

/* sf3d_ext_get_layer_rasters: Project3D::computeCriteria3DMap (project3D.cpp:1896-1947) for layers
 * [first_layer, first_layer + n_layers), e.g. all layers of the water potential as saveModelsState
 * writes them (bin/CRITERIA3D/criteria3DProject.cpp:2275-2301):
 * dst[l][cell] = (float) field value of node(first_layer + l, cell); nodata for cells outside the
 * catchment and for values equal to -9999; SF3D_F_WATER_CONTENT on layer 0 is converted from [m] to
 * [mm] (:1936-1940).  dst is a HOST buffer of n_layers*rows*cols floats. */
uint8_t sf3d_ext_get_layer_rasters(int field, uint32_t first_layer, uint32_t n_layers, float nodata, float *dst);

/* The same maps without blocking the caller (product: the maps are written into a device staging buffer in stream order,
 * i.e. they are the state after every step computed so far, and copied to dst on a second stream while later sf3d_* calls
 * -- the next computeStep -- run; dst should be page-locked host memory, otherwise the copy is staged by the driver and may not
 * overlap).  dst must not be read before sf3d_ext_wait_rasters() has returned; at most two copies are in flight, a third call waits
 * on the device for the oldest.  CPU libraries: the synchronous call, and a no-op wait. */
uint8_t sf3d_ext_get_layer_rasters_async(int field, uint32_t first_layer, uint32_t n_layers, float nodata, float *dst);
uint8_t sf3d_ext_wait_rasters(void);

/* setNodeBoundaryFixedTemperature(i, T[k], depth) for nodes [first, first+count) */
uint8_t sf3d_ext_set_fixed_temperature(uint32_t first, uint32_t count, const double *temperature, double depth);

/* counters since sf3d_initialize (what the reference keeps implicit) */
typedef struct sf3d_counters {
    uint64_t steps;            /* accepted water steps (computeStep calls that returned)   */
    uint64_t tries;            /* passes of the retry loop (cpusolver.cpp:153)             */
    uint64_t approximations;   /* Picard approximations started (cpusolver.cpp:397)        */
    uint64_t sweeps;           /* Jacobi sweeps executed (water.cpp:565)                   */
    uint64_t heat_steps;       /* accepted heat sub-steps                                  */
    uint64_t heat_sweeps;      /* heat linear-solver sweeps                                */
    uint64_t kernel_launches;  /* product only: CUDA kernels launched by the library       */
    double   delta_t_curr;     /* solver deltaTcurr after the last call                    */
    double   last_courant;     /* nodeGrid.CourantWater                                    */
    double   last_mbr;         /* balanceDataCurrentTimeStep.waterMBR                      */
    double   last_mbe;         /* balanceDataCurrentTimeStep.waterMBE                      */
    uint64_t links;            /* existing links (stored off-diagonals of a full assembly) */
    uint64_t heat_cap_hits;    /* heat linear solves that stopped at their sweep cap instead of at the
                                  residual tolerance (cpusolver.cpp:676-700; reference: Gauss-Seidel cap,
                                  product: 4x that cap of Jacobi sweeps) -- SURVEY Appendix B Q6          */
} sf3d_counters;
uint8_t sf3d_ext_get_counters(sf3d_counters *out);
uint8_t sf3d_ext_reset_counters(void);

/* Known-answer entry for the hot kernel: ONE Jacobi sweep (Water::JacobiWaterCPU, water.cpp:565-601) on a
 * caller-supplied system in the reference's compact row layout (MatrixCPU, types_cpu.h:7-13: per row
 * ncols[r] entries, entry 0 = diagonal, then the stored off-diagonals; 11 slots per row).  Rows
 * [0, n_surface) are clamped to x >= z.  Writes x_out and returns the mean norm in *norm.  Independent of
 * the global instance.  The CPU libraries implement it with their own sweep. */
uint8_t sf3d_ext_jacobi_sweep(uint32_t n, uint32_t n_surface, const uint8_t *ncols, const uint32_t *col,
                              const double *val, const double *b, const double *z, const double *x_in,
                              double *x_out, double *norm);

/* Error of the most recent sf3d_compute_step / sf3d_compute_period, then cleared (SF3D_OK when the call
 * succeeded).  The reference's computeStep returns the accepted time step and drops solver->run()'s error code
 * (soilFluxes3D.cpp:1796); this is where a caller can still see it.  Product: SF3D_SOLVER_ERROR when a device
 * or communication fault abandoned the step (e.g. a row-slab peer that did not answer an all-reduce within
 * SF3D_MAILBOX_TIMEOUT_S) -- computeStep then returns the negative sentinel of getDoubleErrorValue instead
 * of a time step and the state is undefined.  CPU libraries: always SF3D_OK. */
uint8_t sf3d_ext_last_error(void);

/* name/version of the implementation behind the ABI ("b200", "oracle", "reference") */
const char *sf3d_ext_backend(void);

/* Restore the solver parameters (types.h:291-315 defaults, deltaTcurr unset) to what a fresh
 * process has.  The reference keeps them in a global solver object that survives
 * cleanSF3D/initializeSF3D (cpusolver.cpp:105-134), so a second catchment in the same process
 * would otherwise start from the previous run's deltaTcurr.  Call before sf3d_initialize. */
uint8_t sf3d_ext_reset_solver(void);

/* Solver::setTimeStep (solver.h:77-86; as written there it ends up assigning the argument unclamped, SURVEY Q10):
 * the time step the next sf3d_compute_step starts from (deltaTcurr).  Together with sf3d_ext_set_field(TOTAL_POTENTIAL)
 * and sf3d_initialize_balance it lets a harness replay the same steps from a saved state. */
uint8_t sf3d_ext_set_time_step(double delta_t);

/* product only: device selection and multi-GPU slab wiring (see DESIGN.md).  The other
 * two libraries return SF3D_PARAMETER_ERROR. */
uint8_t sf3d_ext_set_device(int device);

/* product only: row-slab partition of one catchment over several GPUs, one process per GPU.
 * Each rank initialises its slab (owned DEM rows plus one ghost row per neighbour) as an ordinary
 * catchment, then declares which local nodes are ghosts (recv lists) and which owned nodes the
 * neighbours need (send lists).  The library exchanges x on those lists after every Jacobi sweep
 * and all-reduces the residual, Courant and balance sums (NCCL over NVLink; see DESIGN.md).
 * The 128-byte id is an ncclUniqueId: rank 0 creates it, the harness broadcasts it.  id == NULL: no NCCL
 * communicator; the ranks then talk through peer memory only (sf3d_ext_ipc_* and sf3d_ext_mailbox_* must be wired
 * before the first step), which also works for several ranks sharing one device (used by the tests). */
uint8_t sf3d_ext_comm_unique_id(uint8_t id[128]);
uint8_t sf3d_ext_comm_init(int rank, int world, const uint8_t id[128]);
uint8_t sf3d_ext_comm_finalize(void);
uint8_t sf3d_ext_set_halo(uint32_t n_peers, const int32_t *peers,
                          const uint32_t *send_count, const uint32_t *send_idx,   /* concatenated per peer */
                          const uint32_t *recv_count, const uint32_t *recv_idx,
                          uint64_t n_global_nodes);

/* product only, optional after sf3d_ext_set_halo: the peer-memory transport.  Each rank exports CUDA IPC
 * handles of its two solution buffers (128 bytes) and of a small mailbox (64 bytes); it imports the buffer
 * handles of every neighbour, together with the position of each of its send entries in the neighbour's
 * numbering (the neighbour's recv list), and the mailboxes of ALL other ranks.  With all of them imported
 * (at most 4 neighbours; sf3d_ext_ipc_import fails beyond that) every sweep is one kernel that stores the
 * boundary rows straight into the neighbours' ghost rows over NVLink, and the residual / Courant / balance
 * all-reduces run inside the producing kernels through the mailboxes (deterministic rank-order fold);
 * otherwise the library uses NCCL.  Wire all ranks or none: the choice must be the same on every rank. */
uint8_t sf3d_ext_ipc_export(uint8_t handles[128]);
uint8_t sf3d_ext_ipc_import(int peer, const uint8_t handles[128], uint32_t n, const uint32_t *remote_idx);
uint8_t sf3d_ext_mailbox_export(uint8_t handle[64]);
uint8_t sf3d_ext_mailbox_import(int peer, const uint8_t handle[64]);

/* product only: the cudaStream_t every kernel of the library is launched on (for CUDA-event
 * timing from the harness); NULL in the CPU libraries. */
void *sf3d_ext_stream(void);

/* product only: per-kernel device time, measured with CUDA events on the library's stream
 * around every launch while profiling is enabled (bench.py's roofline figures). */
enum sf3d_kernel {
    SF3D_K_BEGIN_TRY = 0, SF3D_K_NODE_PHASE = 1, SF3D_K_ASSEMBLE = 2, SF3D_K_JACOBI = 3,
    SF3D_K_POST = 4, SF3D_K_ACCEPT = 5, SF3D_K_OTHER = 6,
    SF3D_K_HEAT_COEFFS = 7, SF3D_K_HEAT_FLUX_SNAPSHOT = 8, SF3D_K_HEAT_BOUNDARY = 9, SF3D_K_HEAT_ASSEMBLE = 10,
    SF3D_K_HEAT_JACOBI = 11, SF3D_K_HEAT_POST = 12, SF3D_K_HEAT_ACCEPT = 13, SF3D_K_COMM = 14, SF3D_K_COUNT = 15
};
typedef struct sf3d_kernel_times {
    double   ms[SF3D_K_COUNT];        /* accumulated device time per kernel kind            */
    uint64_t launches[SF3D_K_COUNT];  /* launches per kernel kind                           */
} sf3d_kernel_times;
uint8_t sf3d_ext_profile(int enable);                 /* also resets the accumulators        */
uint8_t sf3d_ext_get_kernel_times(sf3d_kernel_times *out);

#ifdef __cplusplus
}
#endif
#endif /* SF3D_H */
