// sf3d_view.h -- data layout of the soilFluxes3D state in HBM (structure of arrays) and the
// plain-old-data "view" that every kernel receives by value.
//
// Reference layout being replaced: nodesData_t / linkData_t[10] / boundaryData_t / waterData_t /
// heatData_t (agrolib/soilFluxes3D/types.h:136-284) plus the row-pointer ELL matrix MatrixCPU
// (types_cpu.h:7-20).  Here every quantity is one contiguous device array of length N (nodes)
// or 10 x N (link slots, slot-major), so that a warp touching 32 consecutive nodes issues fully
// coalesced 256-byte requests.  Surface nodes occupy [0, nSurface) as in the reference
// (cpusolver.cpp:151,166,413,426).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SF3D_HD __host__ __device__ __forceinline__
#else
#define SF3D_HD inline
#endif

// streaming loads: matrix values, right-hand side and static geometry are read once per pass; mark
// them evict-first so that the 126 MB L2 keeps the gathered vectors (x, K, H) instead
#if defined(__CUDA_ARCH__)
#define SF3D_LDS(p) __ldcs(p)
#else
#define SF3D_LDS(p) (*(p))
#endif

// SF3D_DEVICE_MATH selects the arithmetic variants of the product's device code (powers as exp(y log x), small
// integer powers as multiplications, per-node logarithms of the link means): a few ulp from the reference's
// expressions, far inside the stated tolerances.  -DSF3D_REFERENCE_ROUNDING keeps the reference's expressions
// everywhere; -DSF3D_HOST_DEVICE_MATH compiles the device variants for the host as well (development builds that
// run the row functions on the CPU to check tolerances without a GPU).
#if (defined(__CUDA_ARCH__) || defined(SF3D_HOST_DEVICE_MATH)) && !defined(SF3D_REFERENCE_ROUNDING)
#define SF3D_DEVICE_MATH 1
#endif

// A per-node operand of the logarithmic link means of the heat closures (thermal liquid / vapour conductivity,
// isothermal vapour conductivity, soil heat conductivity).  Device math keeps the value TOGETHER with its natural
// logarithm (16 bytes, one vector load per gather): mean(a, b) = (a - b) / (ln a - ln b) then costs one division per
// link instead of two divisions and a logarithm; the reference-rounding build stores the value only and evaluates
// Math::computeMean as written.  The arrays are allocated with two doubles per node in both builds.
struct alignas(16) SF3DPair { double v, l; };

#define SF3D_NLINK 10           // maxTotalLink, types.h:25
#define SF3D_NODATA (-9999.0)   // commonConstants.h:31

// boundaryType_t values (types.h:98-99)
enum : uint32_t { BT_NONE = 0, BT_RUNOFF = 1, BT_FREE_DRAINAGE = 2, BT_FREE_LATERAL = 3, BT_PRESCRIBED = 4,
                  BT_URBAN = 5, BT_ROAD = 6, BT_CULVERT = 7, BT_HEAT_SURFACE = 8, BT_SOLUTE = 9 };

// meta word per node:  bits 0-3 boundary type | bit 4 surface flag | bits 5-8 numLateralLink |
//                      bits 9-18 link-present mask in SLOT order (slot 0 Up, 1 Down, 2.. Lateral) |
//                      bit 19 ghost flag
#define META_BT(m)        ((m) & 0xFu)
#define META_SURFACE(m)   (((m) >> 4) & 1u)
#define META_NLAT(m)      (((m) >> 5) & 0xFu)
#define META_LINKMASK(m)  (((m) >> 9) & 0x3FFu)
#define META_HAS_SLOT(m, s) (((m) >> (9 + (s))) & 1u)
#define META_GHOST(m)     (((m) >> 19) & 1u)   // halo copy of a node owned by another rank (multi-GPU slabs)

// 16-bit pattern id of a row (see kern_build_patterns): bits 0-14 index the pattern table; bit 15 marks rows the
// interior loop of the multi-GPU sweep skips: ghost rows (id 0xFFFF, never swept) and boundary rows, which the sweep
// computes FIRST so that their values travel to the neighbouring ranks while the interior rows are swept
#define SF3D_PID_MASK     0x7FFFu
#define SF3D_PID_SKIP     0x8000u
#define SF3D_GHOST_PID    0xFFFFu

// Matrix columns are stored in the reference's COLUMN order, which fixes the floating-point
// summation order of the Jacobi row (cpusolver.cpp:352-374): column 0 = Up (slot 0),
// columns 1..8 = Lateral 0..7 (slots 2..9), column 9 = Down (slot 1).
SF3D_HD int sf3d_slot_of_col(int c) { return c == 0 ? 0 : (c == 9 ? 1 : c + 1); }
SF3D_HD int sf3d_col_of_slot(int s) { return s == 0 ? 0 : (s == 1 ? 9 : s - 1); }

// soil horizon record (soilData_t, types.h:104-121) + constants hoisted out of the node loop
struct SoilRec {
    double alpha, n, m, he, Sc, thetaS, thetaR, Ksat, L, organicMatter, clay;
    double invM;        // 1 / m                               (soilPhysics.cpp:186)
    double invSc;       // 1 / Sc                              (soilPhysics.cpp:110)
    double etaClay;     // 1 + 2.6 / sqrt(clay)                (heat.cpp:816)
    double ScPowInvM;   // pow(Sc, 1/m)                        (soilPhysics.cpp:203)
    double tDen;        // 1 - pow(1 - pow(Sc,1/m), m)         (soilPhysics.cpp:206)
};

struct CulvertRec { double width, height, roughness; };   // culvertData_t, types.h:159-164

struct SolverParams {           // SolverParameters, types.h:291-315
    double MBRThreshold, residualTolerance;
    double deltaTmin, deltaTmax, deltaTcurr;
    uint16_t maxApproximationsNumber, maxIterationsNumber;
    uint8_t wrcModel, meanType;
    double lateralVerticalRatio, heatWeightFactor;
    double CourantWaterThreshold, instabilityFactor;
};

// device control block: scalars produced by reductions and the on-device solver state
enum : int { SOLVE_RUNNING = 0, SOLVE_CONVERGED = 1, SOLVE_DIVERGED = 2, SOLVE_MAXITER = 3, SOLVE_COURANT_FAIL = 4,
             SOLVE_COMM_ERROR = 5 };      // a row-slab peer did not answer an all-reduce: never a numerical event
struct Ctrl {
    double courantMax;      // nodeGrid.CourantWater
    double storage;         // sum theta*V            (water.cpp:71-90)
    double sinkSum;         // sum waterFlow*dt       (water.cpp:130-140)
    double lastNorm;        // JacobiWaterCPU return value of the last sweep
    double bestNorm;        // solveLinearSystem bestErrorNorm
    double heatCourantMax;  // updateBoundaryHeatData
    double heatStorage, heatSinkSum;
    double boundarySum;     // getTotalBoundaryWaterFlow
    int    status;          // SOLVE_*
    int    sweeps;          // sweeps executed in the current solve
    unsigned int ticket;    // last-block election counter
    int    commError;       // multi-GPU: set when a mailbox all-reduce timed out; read_ctrl turns it into a DeviceError
    double red[4];          // multi-GPU: local reductions handed to the all-reduce before the rule is applied
    // multi-GPU: device-side clocks of the in-kernel all-reduces (globaltimer, ns): time between the election of the
    // last block (all rows of this rank done) and the end of the all-reduce = wait for the slowest rank + NVLink
    // latency; summed over the all-reduces executed, with their count.  Reported as kernel kind "comm".
    unsigned long long commNs, commCount;
};

struct SF3DView {
    uint32_t N, Ns;                 // nodes, surface nodes (local, ghosts included)
    uint32_t world;                 // number of ranks sharing the catchment (1 = single GPU)
    double   nGlobal;               // owned nodes summed over ranks (= N when world == 1)
    // flags (simulationFlags_t, types.h:188-197)
    int computeHeat, computeHeatVapor, computeHeatAdvection, hfSaveMode;
    // solver parameters needed on device
    int wrcModel, meanType;
    double lvRatio, heatWF;

    // topology
    double *x, *y, *z, *size;
    uint32_t *meta;                 // packed, see META_*
    uint16_t *tab;                  // soil-table / surface-table index
    // boundary
    double *bSlope, *bSize, *bRate, *bSum, *bPresc;
    // links, slot-major: [slot*N + i]
    uint32_t *lidx;
    double *larea, *lflow;
    double *lgeom;                  // static link geometry, COLUMN-major (see sf3d_link_geom)
    // water state
    double *H, *oldH, *bestH, *Se, *SeOld, *K, *wFlow, *sink, *pond;
    // linear system, COLUMN-major: [col*N + i]; mcol is static
    uint32_t *mcol;
    // pattern-compressed column indices: mcol[c][i] == i + pattern[pid[i]*10 + c] for every node
    // (verified bit-exactly at finalize).  pattern is null when the graph has too many distinct link patterns
    // (or SF3D_EXPLICIT_INDEX is set); pid is set in either case, since it also carries the row class (see
    // SF3D_PID_SKIP).  Both null only in single-rank views without a pattern build.
    const uint16_t *pid;
    const int32_t *pattern;
    uint32_t hotPid;                // the most frequent pattern (interior nodes) and its offsets, held in
    int32_t hotOff[SF3D_NLINK];     // kernel parameters so that the common case needs no table load
    double *mval;
    double *b, *cap, *x0, *x1;
    // tables
    const SoilRec *soil;
    const double *rough;
    const CulvertRec *culverts;     // null when no culvert is defined
    const uint32_t *culvertOf;      // [Ns] 1 + index into culverts; 0 = the node has no culvert record
    // heat (null when !computeHeat)
    double *T, *oldT, *hFlux, *hSink;
    double *hbHeightWind, *hbHeightT, *hbRough, *hbAero, *hbSoilCond, *hbT, *hbRH, *hbWind, *hbNetIrr;
    double *hbSens, *hbLat, *hbRad, *hbAdv, *hbFixT, *hbFixDepth;
    double *lwFlux, *lvFlux;        // per link, slot-major (float-rounded values, heat.cpp:126-127)
    double *lfluxes;                // [type][slot][i], types allocated per hfSaveMode
    double *hdiag;                  // heat matrix diagonal (kept, cpusolver.cpp:561-567)
    // per-node coefficients the reference re-evaluates for both ends of every link (same arguments, same
    // value): thermal / isothermal vapour conductivity and soil heat conductivity, computed once per node
    double *hTVK, *hIVK, *hCond;    // (each of these five link operands: SF3DPair per node under device math, see above)
    // water-side coupling, stored by the node phase: mean temperature and thermal liquid conductivity
    // (mean T, current psi); heat side: thermal liquid conductivity (T, sub-step averaged psi)
    double *hTm, *hTLK, *hTLKh;
    double *hInv;                   // water side: the row's thermal liquid / vapour flux sum (invariantFluxes, water.cpp:329-340)
    double *hHs, *hPsiAvg;          // heat side, per sub-step: getNodeH_fromTimeSteps and the sub-step averaged matric head
    double *hPress;                 // static: pressureFromAltitude(z), heat.cpp:1117
    double *ldist3;                 // static per link, slot-major: nodeDistance3D (soilPhysics.cpp:331-335); device math
                                    // stores interfaceArea / nodeDistance3D instead (every use is flux density x area / distance)
    // control / reduction scratch
    Ctrl *ctrl;
    double *partA, *partB;          // per-block partials
};
