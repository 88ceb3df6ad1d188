// sf3d_capi.cpp -- the C ABI of include/sf3d.h for the B200 product.
//
// Role: the reference's soilFluxes3D.cpp (global nodeGrid + scalar setters/getters) with the
// state living in HBM.  Scalar setters/getters work on lazily allocated host mirrors; a mirror
// is pushed to the device in one copy before the next kernel needs it and pulled in one copy
// the first time a getter asks after the device changed it (SURVEY 3.5).  Bulk extensions move
// whole ranges and never allocate host mirrors.  Validation and return codes follow the
// reference function of the same name (file:line cited at each function).
#include <float.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <thread>
#include <vector>
#include "sf3d.h"
#include "sf3d_engine.h"
#include "sf3d_rows_heat.h"

using namespace sf3d;

namespace {

template <class T>
struct Mirror {
    T *d = nullptr;
    T *h = nullptr;
    size_t n = 0;
    bool hostNewer = false, devNewer = false;

    void alloc(size_t count) { n = count; d = (T *)dev_alloc(count * sizeof(T)); }
    void release() { dev_free(d); free(h); d = h = nullptr; n = 0; hostNewer = devNewer = false; }
    T *sync_host()
    {
        if (!h) { h = (T *)calloc(n ? n : 1, sizeof(T)); if (!h) throw DeviceError{-2, "host alloc", "Mirror"}; }
        if (devNewer) { d2h(h, d, n * sizeof(T)); devNewer = false; }
        return h;
    }
    const T *ro() { return sync_host(); }
    T *rw() { T *p = sync_host(); hostNewer = true; return p; }
    void push() { if (hostNewer) { h2d(d, h, n * sizeof(T)); hostNewer = false; } }
    void dev_written() { devNewer = true; }     // call after push()
};

struct State {
    bool initialized = false;
    bool water = true, heat = false, solutes = false, heatVapor = false, heatAdvection = false;
    uint8_t hfMode = 0;
    uint32_t N = 0, Ns = 0;
    double nGlobal = 0.;                 // owned nodes over all ranks (multi-GPU slabs)

    std::vector<SoilRec> soils;
    std::vector<std::pair<uint16_t, uint8_t>> soilKeys;   // (soilNumber, horizonNumber) of each record
    std::vector<std::vector<uint16_t>> soil1D;
    std::vector<double> rough;
    std::vector<CulvertRec> culverts;
    bool tablesDirty = true, topoDirty = true;
    SoilRec *dSoil = nullptr; double *dRough = nullptr; CulvertRec *dCulv = nullptr;
    size_t dSoilCap = 0, dRoughCap = 0, dCulvCap = 0;

    Mirror<double> x, y, z, size, bSlope, bSize, bRate, bSum, bPresc;
    Mirror<uint32_t> meta, lidx, culvertOf;
    Mirror<uint16_t> tab;
    Mirror<double> larea, lflow;
    Mirror<double> H, oldH, Se, K, sink, pond;
    // heat (allocated when isComputeHeat)
    Mirror<double> T, oldT, hSink;
    Mirror<double> hbHeightWind, hbHeightT, hbRough, hbAero, hbSoilCond, hbT, hbRH, hbWind, hbNetIrr,
                   hbSens, hbLat, hbRad, hbAdv, hbFixT, hbFixDepth;
    Mirror<double> lfluxes;               // [type][slot][node]; 1 type (HeatTotal) unless save mode All (9)
    int hfTypesAllocated = 0;
    double *hFlux = nullptr, *lwFlux = nullptr, *lvFlux = nullptr, *hdiag = nullptr, *hTVK = nullptr, *hIVK = nullptr, *hCond = nullptr,
           *hTm = nullptr, *hTLK = nullptr, *hTLKh = nullptr, *hPress = nullptr, *ldist3 = nullptr, *hHs = nullptr, *hPsiAvg = nullptr, *hInv = nullptr;
    // device-only
    double *bestH = nullptr, *SeOld = nullptr, *wFlow = nullptr, *lgeom = nullptr, *mval = nullptr,
           *b = nullptr, *cap = nullptr, *x0 = nullptr, *x1 = nullptr, *partA = nullptr, *partB = nullptr,
           *scratch = nullptr;
    uint32_t *mcol = nullptr;
    uint16_t *pid = nullptr; int32_t *pattern = nullptr; bool patternsOk = false;
    void *overlapStage[2] = {nullptr, nullptr}; size_t overlapStageBytes[2] = {0, 0}; int overlapSlot = 0;
    uint32_t hotPid = 0; int32_t hotOff[SF3D_NLINK] = {0};
    Ctrl *ctrl = nullptr;
    // raster side of a graph built by sf3d_ext_build_grid (kept for the raster-facing forcing / output calls)
    RasterDev raster{};
    int32_t *rasterRank = nullptr;
    void *rasterStage = nullptr; size_t rasterStageBytes = 0;     // device staging for forcing / output rasters

    Engine eng;
};

State S;
SolverParams g_params = default_params();       // survives cleanSF3D like the global CPUSolverObject
bool g_useLineal = false; int g_linealMethod = 0;
int g_device = 0;

double err_value(uint8_t code)                     // getDoubleErrorValue, types.h:42-64
{
    switch (code)
    {
        case SF3D_OK: return 0;
        case SF3D_INDEX_ERROR: return -1111;
        case SF3D_MEMORY_ERROR: return -2222;
        case SF3D_TOPOGRAPHY_ERROR: return -3333;
        case SF3D_BOUNDARY_ERROR: return -4444;
        case SF3D_MISSING_DATA_ERROR: return -9999;
        case SF3D_PARAMETER_ERROR: return -7777;
        default: return -1111;
    }
}

void fill_view()
{
    SF3DView &v = S.eng.v;
    memset(&v, 0, sizeof v);
    v.N = S.N; v.Ns = S.Ns;
    v.world = (uint32_t)comm_world();
    v.nGlobal = (v.world > 1 && S.nGlobal > 0.) ? S.nGlobal : (double)S.N;
    v.computeHeat = S.heat; v.computeHeatVapor = S.heatVapor; v.computeHeatAdvection = S.heatAdvection;
    v.hfSaveMode = S.hfMode;
    v.wrcModel = g_params.wrcModel; v.meanType = g_params.meanType;
    v.lvRatio = g_params.lateralVerticalRatio; v.heatWF = g_params.heatWeightFactor;
    v.x = S.x.d; v.y = S.y.d; v.z = S.z.d; v.size = S.size.d; v.meta = S.meta.d; v.tab = S.tab.d;
    v.bSlope = S.bSlope.d; v.bSize = S.bSize.d; v.bRate = S.bRate.d; v.bSum = S.bSum.d; v.bPresc = S.bPresc.d;
    v.lidx = S.lidx.d; v.larea = S.larea.d; v.lflow = S.lflow.d; v.lgeom = S.lgeom;
    v.H = S.H.d; v.oldH = S.oldH.d; v.bestH = S.bestH; v.Se = S.Se.d; v.SeOld = S.SeOld; v.K = S.K.d;
    v.wFlow = S.wFlow; v.sink = S.sink.d; v.pond = S.pond.d;
    v.mcol = S.mcol; v.pid = S.pid; v.pattern = S.patternsOk ? S.pattern : nullptr; v.mval = S.mval;
    v.hotPid = S.hotPid; memcpy(v.hotOff, S.hotOff, sizeof v.hotOff); v.b = S.b; v.cap = S.cap; v.x0 = S.x0; v.x1 = S.x1;
    v.soil = S.dSoil; v.rough = S.dRough;
    v.culverts = S.culverts.empty() ? nullptr : S.dCulv;
    v.culvertOf = S.culverts.empty() ? nullptr : S.culvertOf.d;
    v.ctrl = S.ctrl; v.partA = S.partA; v.partB = S.partB;
    if (S.heat)
    {
        v.T = S.T.d; v.oldT = S.oldT.d; v.hFlux = S.hFlux; v.hSink = S.hSink.d;
        v.hbHeightWind = S.hbHeightWind.d; v.hbHeightT = S.hbHeightT.d; v.hbRough = S.hbRough.d; v.hbAero = S.hbAero.d;
        v.hbSoilCond = S.hbSoilCond.d; v.hbT = S.hbT.d; v.hbRH = S.hbRH.d; v.hbWind = S.hbWind.d; v.hbNetIrr = S.hbNetIrr.d;
        v.hbSens = S.hbSens.d; v.hbLat = S.hbLat.d; v.hbRad = S.hbRad.d; v.hbAdv = S.hbAdv.d;
        v.hbFixT = S.hbFixT.d; v.hbFixDepth = S.hbFixDepth.d;
        v.lwFlux = S.lwFlux; v.lvFlux = S.lvFlux; v.lfluxes = S.lfluxes.d; v.hdiag = S.hdiag;
        v.hTVK = S.hTVK; v.hIVK = S.hIVK; v.hCond = S.hCond;
        v.hTm = S.hTm; v.hTLK = S.hTLK; v.hTLKh = S.hTLKh; v.hPress = S.hPress; v.ldist3 = S.ldist3;
        v.hHs = S.hHs; v.hPsiAvg = S.hPsiAvg; v.hInv = S.hInv;
    }
}

Mirror<double> *heat_boundary_mirrors[15];
void collect_heat_mirrors()
{
    Mirror<double> *m[15] = {&S.hbHeightWind, &S.hbHeightT, &S.hbRough, &S.hbAero, &S.hbSoilCond, &S.hbT, &S.hbRH, &S.hbWind,
                             &S.hbNetIrr, &S.hbSens, &S.hbLat, &S.hbRad, &S.hbAdv, &S.hbFixT, &S.hbFixDepth};
    for (int k = 0; k < 15; ++k) heat_boundary_mirrors[k] = m[k];
}

void upload_tables()
{
    if (!S.tablesDirty) return;
    if (S.soils.size() > S.dSoilCap)
    {
        dev_free(S.dSoil);
        S.dSoilCap = std::max<size_t>(64, S.soils.size() * 2);
        S.dSoil = (SoilRec *)dev_alloc(S.dSoilCap * sizeof(SoilRec));
    }
    if (!S.soils.empty()) h2d(S.dSoil, S.soils.data(), S.soils.size() * sizeof(SoilRec));
    if (S.rough.size() > S.dRoughCap)
    {
        dev_free(S.dRough);
        S.dRoughCap = std::max<size_t>(64, S.rough.size() * 2);
        S.dRough = (double *)dev_alloc(S.dRoughCap * sizeof(double));
    }
    if (!S.rough.empty()) h2d(S.dRough, S.rough.data(), S.rough.size() * sizeof(double));
    if (S.culverts.size() > S.dCulvCap)
    {
        dev_free(S.dCulv);
        S.dCulvCap = std::max<size_t>(16, S.culverts.size() * 2);
        S.dCulv = (CulvertRec *)dev_alloc(S.dCulvCap * sizeof(CulvertRec));
    }
    if (!S.culverts.empty()) h2d(S.dCulv, S.culverts.data(), S.culverts.size() * sizeof(CulvertRec));
    S.tablesDirty = false;
}

// everything the kernels read must be current on the device
uint8_t sync_to_device(bool finalizeTopology = true)
{
    // anything set on the host since the last step that the next try's first pass depends on: that pass must run
    if (S.tablesDirty || S.topoDirty || S.H.hostNewer || S.oldH.hostNewer || S.Se.hostNewer || S.z.hostNewer || S.size.hostNewer
        || S.tab.hostNewer || S.meta.hostNewer)
        S.eng.tryPrepared = false;
    upload_tables();
    S.x.push(); S.y.push(); S.z.push(); S.size.push(); S.meta.push(); S.tab.push();
    S.bSlope.push(); S.bSize.push(); S.bRate.push(); S.bSum.push(); S.bPresc.push();
    S.lidx.push(); S.larea.push(); S.lflow.push(); S.culvertOf.push();
    S.H.push(); S.oldH.push(); S.Se.push(); S.K.push(); S.sink.push(); S.pond.push();
    if (S.heat)
    {
        S.T.push(); S.oldT.push(); S.hSink.push(); S.lfluxes.push();
        collect_heat_mirrors();
        for (Mirror<double> *m : heat_boundary_mirrors) m->push();
    }
    fill_view();
    if (S.topoDirty && finalizeTopology)
    {
        int ok = 1;
        S.patternsOk = false;
        fill_view();
        k_link_geometry(S.eng.v, &ok);
        if (S.heat) k_heat_geometry(S.eng.v);
        S.patternsOk = k_build_patterns(S.eng.v, S.pid, S.pattern, &S.hotPid, S.hotOff) && getenv("SF3D_EXPLICIT_INDEX") == nullptr;
        comm_mark_boundary(S.pid);
        fill_view();
        S.topoDirty = false;
        if (!ok)
        {
            fprintf(stderr, "[sf3d_b200] topology error: surface nodes must occupy indices [0, nrSurfaceNodes) "
                            "(the reference solver assumes it: cpusolver.cpp:151,166,413,426)\n");
            return SF3D_TOPOGRAPHY_ERROR;
        }
    }
    return SF3D_OK;
}

void step_wrote_device()
{
    S.H.dev_written(); S.oldH.dev_written(); S.Se.dev_written(); S.K.dev_written();
    S.bRate.dev_written(); S.bSum.dev_written(); S.lflow.dev_written();
    if (S.heat)
    {
        S.T.dev_written(); S.oldT.dev_written(); S.lfluxes.dev_written();
        S.hbAero.dev_written(); S.hbSoilCond.dev_written(); S.hbSens.dev_written(); S.hbLat.dev_written();
        S.hbRad.dev_written(); S.hbAdv.dev_written();
    }
}

// host-side physics for the scalar setters (same row functions, compiled for the host)
double host_se_from_theta(const SoilRec &s, double theta)          // soilPhysics.cpp:123-134
{
    if (theta >= s.thetaS) return 1.;
    if (theta < s.thetaR) return 0.;
    return (theta - s.thetaR) / (s.thetaS - s.thetaR);
}
double host_psi_from_se(const SoilRec &s, double Se)               // Soil::computeNodePsi, soilPhysics.cpp:141-158
{
    double temp;
    if (g_params.wrcModel == 0) temp = pow(1. / Se, 1. / s.m) - 1.;
    else if (g_params.wrcModel == 1) temp = pow(1. / (Se * s.Sc), 1. / s.m) - 1;
    else return SF3D_NODATA;
    return (1. / s.alpha) * pow(temp, 1. / s.n);
}
const SoilRec &node_soil(uint32_t i) { return S.soils[S.tab.ro()[i]]; }
bool is_surface(uint32_t i) { return META_SURFACE(S.meta.ro()[i]) != 0; }
uint32_t node_bt(uint32_t i) { return META_BT(S.meta.ro()[i]); }
double host_node_K(uint32_t i, double Se) { return sf3d_mualem(node_soil(i), g_params.wrcModel, Se); }

#define REQUIRE_INIT_E()  do { if (!S.initialized) return SF3D_MEMORY_ERROR; } while (0)
#define REQUIRE_INDEX_E(i) do { if ((i) >= S.N) return SF3D_INDEX_ERROR; } while (0)
#define REQUIRE_INIT_D()  do { if (!S.initialized) return err_value(SF3D_MEMORY_ERROR); } while (0)
#define REQUIRE_INDEX_D(i) do { if ((i) >= S.N) return err_value(SF3D_INDEX_ERROR); } while (0)

uint8_t g_lastStepError = SF3D_OK;              // sf3d_ext_last_error

template <class F>
auto guarded(F &&f, decltype(f()) onError) -> decltype(f())
{
    try { return f(); }
    catch (const DeviceError &e)
    {
        fprintf(stderr, "[sf3d_b200] device error in %s: %s\n", e.where, e.what);
        g_lastStepError = SF3D_SOLVER_ERROR;
        return onError;
    }
}

void release_all()
{
    S.x.release(); S.y.release(); S.z.release(); S.size.release(); S.bSlope.release(); S.bSize.release();
    S.bRate.release(); S.bSum.release(); S.bPresc.release(); S.meta.release(); S.lidx.release();
    S.culvertOf.release(); S.tab.release(); S.larea.release(); S.lflow.release();
    S.H.release(); S.oldH.release(); S.Se.release(); S.K.release(); S.sink.release(); S.pond.release();
    S.T.release(); S.oldT.release(); S.hSink.release(); S.lfluxes.release();
    collect_heat_mirrors();
    for (Mirror<double> *m : heat_boundary_mirrors) m->release();
    { double **hd[] = {&S.hFlux, &S.lwFlux, &S.lvFlux, &S.hdiag, &S.hTVK, &S.hIVK, &S.hCond, &S.hTm, &S.hTLK, &S.hTLKh, &S.hPress, &S.ldist3, &S.hHs, &S.hPsiAvg, &S.hInv}; for (double **p : hd) { dev_free(*p); *p = nullptr; } }
    S.hfTypesAllocated = 0;
    double **devOnly[] = {&S.bestH, &S.SeOld, &S.wFlow, &S.lgeom, &S.mval, &S.b, &S.cap, &S.x0, &S.x1,
                          &S.partA, &S.partB, &S.scratch};
    for (double **p : devOnly) { dev_free(*p); *p = nullptr; }
    dev_free(S.mcol); S.mcol = nullptr;
    dev_free(S.pid); S.pid = nullptr; dev_free(S.pattern); S.pattern = nullptr; S.patternsOk = false;
    dev_free(S.ctrl); S.ctrl = nullptr;
    dev_free(S.rasterRank); S.rasterRank = nullptr; S.raster = RasterDev{};
    dev_free(S.rasterStage); S.rasterStage = nullptr; S.rasterStageBytes = 0;
    // overlapped map downloads still in flight read these buffers: wait for them first (a device error here is left to the
    // next call that touches the device)
    try { overlap_sync(); } catch (const DeviceError &) {}
    for (int k = 0; k < 2; ++k) { dev_free(S.overlapStage[k]); S.overlapStage[k] = nullptr; S.overlapStageBytes[k] = 0; }
}

void *raster_stage(size_t bytes)
{
    if (S.rasterStageBytes < bytes)
    {
        dev_free(S.rasterStage); S.rasterStage = nullptr; S.rasterStageBytes = 0;
        S.rasterStage = dev_alloc(bytes); S.rasterStageBytes = bytes;
    }
    return S.rasterStage;
}

double *scratch_buffer()
{
    if (!S.scratch) S.scratch = (double *)dev_alloc((size_t)S.N * sizeof(double));
    return S.scratch;
}

}  // namespace

extern "C" {

// ---- initializeSF3D (soilFluxes3D.cpp:49-178) ------------------------------------------------
uint8_t sf3d_initialize(uint32_t nrNodes, uint32_t nrSurfaceNodes, uint8_t nrLateralLinks,
                        int isComputeWater, int isComputeHeat, int isComputeSolutes, uint8_t hfMode)
{
    return guarded([&]() -> uint8_t {
        uint8_t rc = sf3d_clean();
        if (rc) return rc;
        dev_select(g_device);
        S.water = isComputeWater != 0; S.heat = isComputeHeat != 0; S.solutes = isComputeSolutes != 0;
        S.heatVapor = S.heatAdvection = false; S.hfMode = 0;
        if (S.heat) { S.heatVapor = true; S.heatAdvection = true; S.hfMode = hfMode; }
        S.N = nrNodes; S.Ns = nrSurfaceNodes; S.nGlobal = 0.;
        comm_clear_halo();
        if (nrLateralLinks > SF3D_MAX_LATERAL_LINK) return SF3D_PARAMETER_ERROR;

        const size_t N = nrNodes, L = (size_t)SF3D_NLINK * N;
        S.x.alloc(N); S.y.alloc(N); S.z.alloc(N); S.size.alloc(N); S.meta.alloc(N); S.tab.alloc(N);
        S.bSlope.alloc(N); S.bSize.alloc(N); S.bRate.alloc(N); S.bSum.alloc(N); S.bPresc.alloc(N);
        S.lidx.alloc(L); S.larea.alloc(L); S.lflow.alloc(L);
        S.H.alloc(N); S.oldH.alloc(N); S.Se.alloc(N); S.K.alloc(N); S.sink.alloc(N); S.pond.alloc(nrSurfaceNodes);
        S.culvertOf.alloc(nrSurfaceNodes);
        S.bestH = (double *)dev_alloc(N * 8); S.SeOld = (double *)dev_alloc(N * 8); S.wFlow = (double *)dev_alloc(N * 8);
        S.lgeom = (double *)dev_alloc(L * 8); S.mval = (double *)dev_alloc(L * 8); S.mcol = (uint32_t *)dev_alloc(L * 4);
        S.pid = (uint16_t *)dev_alloc(N * 2); S.pattern = (int32_t *)dev_alloc(pattern_table_bytes());
        S.b = (double *)dev_alloc(N * 8); S.cap = (double *)dev_alloc(N * 8);
        S.x0 = (double *)dev_alloc(N * 8); S.x1 = (double *)dev_alloc(N * 8);
        const size_t nb = (size_t)std::max(reduce_blocks(0xFFFFFFFFu), wide_blocks(0xFFFFFFFFu));
        S.partA = (double *)dev_alloc(nb * 8); S.partB = (double *)dev_alloc(nb * 8);
        S.ctrl = (Ctrl *)dev_alloc(sizeof(Ctrl));
        if (S.heat)
        {
            S.T.alloc(N); S.oldT.alloc(N); S.hSink.alloc(N);
            collect_heat_mirrors();
            for (Mirror<double> *m : heat_boundary_mirrors) m->alloc(N);
            S.hFlux = (double *)dev_alloc(N * 8); S.hdiag = (double *)dev_alloc(N * 8);
            // link operands of the logarithmic means: value + logarithm per node (SF3DPair, sf3d_view.h)
            S.hTVK = (double *)dev_alloc(N * 16); S.hIVK = (double *)dev_alloc(N * 16); S.hCond = (double *)dev_alloc(N * 16);
            S.hTm = (double *)dev_alloc(N * 8); S.hTLK = (double *)dev_alloc(N * 16); S.hTLKh = (double *)dev_alloc(N * 16);
            S.hHs = (double *)dev_alloc(N * 8); S.hPsiAvg = (double *)dev_alloc(N * 8); S.hInv = (double *)dev_alloc(N * 8);
            S.hPress = (double *)dev_alloc(N * 8); S.ldist3 = (double *)dev_alloc(L * 8);
            S.lwFlux = (double *)dev_alloc(L * 8); S.lvFlux = (double *)dev_alloc(L * 8);
            S.hfTypesAllocated = (S.hfMode == 2) ? 9 : 1;
            S.lfluxes.alloc((size_t)S.hfTypesAllocated * L);
        }

        S.tablesDirty = S.topoDirty = true;
        S.initialized = true;

        // CPUSolver::initialize (cpusolver.cpp:25-31)
        if (g_params.deltaTcurr == SF3D_NODATA) g_params.deltaTcurr = g_params.deltaTmax;
        S.eng = Engine{};
        S.eng.p = &g_params;
        S.eng.computeWater = S.water;
        S.eng.computeHeat = S.heat;
        S.eng.tryPrepared = false;
        fill_view();
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- initializeBalance (soilFluxes3D.cpp:184-197) ---------------------------------------------
uint8_t sf3d_initialize_balance(void)
{
    return guarded([&]() -> uint8_t {
        if (!S.initialized) return SF3D_MEMORY_ERROR;         // water.cpp:54-55
        uint8_t rc = sync_to_device();
        if (rc) return rc;
        S.eng.initializeWaterBalance();
        S.lflow.dev_written(); S.bSum.dev_written(); S.Se.dev_written();
        if (S.heat) S.eng.initializeHeatBalance();            // soilFluxes3D.cpp:191-192
        else S.eng.wholePeriod.heatMBR = 1.;                  // soilFluxes3D.cpp:194
        return SF3D_OK;
    }, (uint8_t)SF3D_SOLVER_ERROR);
}

// ---- cleanSF3D (soilFluxes3D.cpp:218-304) -------------------------------------------------------
uint8_t sf3d_clean(void)
{
    if (!S.initialized) return SF3D_OK;
    release_all();
    S.initialized = false;
    S.soils.clear(); S.soilKeys.clear(); S.rough.clear();               // :295-296 (soil1DIndices and culvertList are not cleared)
    S.tablesDirty = true;
    return SF3D_OK;
}

uint8_t sf3d_initialize_heat_flag(uint8_t saveModeHeat, int adv, int lat)     // soilFluxes3D.cpp:325-332
{
    S.hfMode = saveModeHeat; S.heatAdvection = adv != 0; S.heatVapor = lat != 0;
    if (S.initialized && S.heat && S.hfMode == 2 && S.hfTypesAllocated < 9)
        return guarded([&]() -> uint8_t {
            S.lfluxes.release();
            S.hfTypesAllocated = 9;
            S.lfluxes.alloc((size_t)9 * SF3D_NLINK * S.N);
            return SF3D_OK;
        }, (uint8_t)SF3D_MEMORY_ERROR);
    return SF3D_OK;
}

uint32_t sf3d_set_threads_number(uint32_t nrThreads)                           // soilFluxes3D.cpp:340-361
{
    // Same clamping and return value as the reference; the product's parallelism is the GPU's.
    uint32_t hw = std::thread::hardware_concurrency();
    if (nrThreads < 1 || nrThreads > hw) nrThreads = hw;
    return nrThreads;
}
void sf3d_set_use_lineal(int value) { g_useLineal = value != 0; }              // accepted, unused (SURVEY section 2 row 8)
void sf3d_set_lineal_method(int value) { g_linealMethod = value; }


// ---- setSoilProperties (soilFluxes3D.cpp:395-449) -------------------------------------------------
uint8_t sf3d_set_soil_properties(uint16_t nrSoil, uint8_t nrHorizon, double VG_alpha, double VG_n, double VG_m,
                                 double VG_he, double thetaR, double thetaS, double kSat, double MualemL,
                                 double organicMatter, double clay)
{
    if (VG_alpha <= 0 || VG_n <= 1.0 || VG_m <= 0.0 || VG_m >= 1.0 || VG_he < 0.0 || kSat <= 0.0
        || thetaR < 0.0 || thetaR >= 1.0 || thetaS <= 0.0 || thetaS > 1.0 || thetaR > thetaS)
        return SF3D_PARAMETER_ERROR;
    for (const auto &key : S.soilKeys)                                  // :410-412 already defined
        if (key.first == nrSoil && key.second == nrHorizon) return SF3D_PARAMETER_ERROR;
    if (S.soils.size() > 65535) return SF3D_MEMORY_ERROR;               // :415-418

    SoilRec r{};
    r.alpha = VG_alpha; r.n = VG_n; r.m = VG_m; r.he = VG_he;
    r.Sc = pow(1. + pow(VG_alpha * VG_he, VG_n), -VG_m);                // :428
    r.thetaR = thetaR; r.thetaS = thetaS; r.Ksat = kSat; r.L = MualemL;
    r.organicMatter = organicMatter; r.clay = clay;
    r.invM = 1.0 / r.m;
    r.invSc = 1.0 / r.Sc;
    r.etaClay = 1. + 2.6 / sqrt(r.clay);
    r.ScPowInvM = pow(r.Sc, r.invM);
    r.tDen = 1.0 - pow(1.0 - r.ScPowInvM, r.m);

    if (nrSoil >= S.soil1D.size()) S.soil1D.resize((size_t)nrSoil + 1);
    if (nrHorizon >= S.soil1D[nrSoil].size()) S.soil1D[nrSoil].resize((size_t)nrHorizon + 1);
    S.soils.push_back(r);
    S.soilKeys.emplace_back(nrSoil, nrHorizon);
    S.soil1D[nrSoil][nrHorizon] = (uint16_t)(S.soils.size() - 1);
    S.tablesDirty = true;
    return SF3D_OK;
}

// ---- setSurfaceProperties (soilFluxes3D.cpp:457-467) --------------------------------------------------
uint8_t sf3d_set_surface_properties(uint16_t surfaceIndex, double roughness)
{
    if (roughness < 0) return SF3D_PARAMETER_ERROR;
    if (surfaceIndex >= S.rough.size()) S.rough.resize((size_t)surfaceIndex + 1);
    S.rough[surfaceIndex] = roughness;
    S.tablesDirty = true;
    return SF3D_OK;
}

// ---- setNumericalParameters (soilFluxes3D.cpp:474-520) ------------------------------------------------
uint8_t sf3d_set_numerical_parameters(double minDeltaT, double maxDeltaT, uint16_t maxIterationNumber,
                                      uint16_t maxApproximationsNumber, uint8_t tolExp, uint8_t mbrExp)
{
    if (minDeltaT < 0.01) minDeltaT = 0.01;
    if (minDeltaT > 3600.) minDeltaT = 3600.;
    if (maxDeltaT < 60) maxDeltaT = 60;
    if (maxDeltaT > 3600.) maxDeltaT = 3600.;
    if (maxDeltaT < minDeltaT) maxDeltaT = minDeltaT;
    if (maxIterationNumber < 20) maxIterationNumber = 20;
    if (maxIterationNumber > 1000) maxIterationNumber = 1000;
    if (maxApproximationsNumber < 1) maxApproximationsNumber = 1;
    if (maxApproximationsNumber > 50) maxApproximationsNumber = 50;
    if (tolExp < 5) tolExp = 5;
    if (tolExp > 12) tolExp = 12;
    if (mbrExp < 1) mbrExp = 1;
    if (mbrExp > 9) mbrExp = 9;
    g_params.MBRThreshold = pow(10.0, -mbrExp);
    g_params.residualTolerance = pow(10.0, -tolExp);
    g_params.deltaTmin = minDeltaT;
    g_params.deltaTmax = maxDeltaT;
    // deltaTcurr is passed through unchanged (:514)
    g_params.maxApproximationsNumber = maxApproximationsNumber;
    g_params.maxIterationsNumber = maxIterationNumber;
    return SF3D_OK;
}

// ---- setHydraulicProperties (soilFluxes3D.cpp:531-548) ------------------------------------------------
uint8_t sf3d_set_hydraulic_properties(uint8_t wrc, uint8_t meanType, float ratio)
{
    if ((ratio < 0.1) || (ratio > 100)) return SF3D_PARAMETER_ERROR;
    g_params.wrcModel = wrc;
    g_params.meanType = meanType;
    g_params.lateralVerticalRatio = ratio;       // float -> double, as SolverParametersPartial does
    S.topoDirty = true;                          // the static link factors fold the ratio in
    return SF3D_OK;
}

// ---- setNodeBoundary (soilFluxes3D.cpp:689-725) ---------------------------------------------------------
static uint8_t set_node_boundary_unchecked(uint32_t i, uint8_t bt, double slope, double bArea)
{
    uint32_t *meta = S.meta.rw();
    meta[i] = (meta[i] & ~0xFu) | (bt & 0xFu);
    if (bt == BT_NONE) return SF3D_OK;
    S.bSlope.rw()[i] = slope;
    S.bSize.rw()[i] = bArea;
    if (S.water)
    {
        S.bRate.rw()[i] = 0.;
        S.bSum.rw()[i] = 0.;
        S.bPresc.rw()[i] = SF3D_NODATA;
    }
    if (S.heat)                                   // soilFluxes3D.cpp:705-722
    {
        collect_heat_mirrors();
        for (Mirror<double> *m : heat_boundary_mirrors) m->rw()[i] = SF3D_NODATA;
        S.hbRad.rw()[i] = 0.; S.hbLat.rw()[i] = 0.; S.hbSens.rw()[i] = 0.; S.hbAdv.rw()[i] = 0.;
    }
    return SF3D_OK;
}
uint8_t sf3d_set_node_boundary(uint32_t nodeIndex, uint8_t boundaryType, double slope, double boundaryArea)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);       // (the reference has no checks here)
        return set_node_boundary_unchecked(nodeIndex, boundaryType, slope, boundaryArea);
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- setCulvert (soilFluxes3D.cpp:551-588) ---------------------------------------------------------------
uint8_t sf3d_set_culvert(uint32_t nodeIndex, double roughness, double slope, double width, double height)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (nodeIndex >= S.N || !is_surface(nodeIndex) || nodeIndex >= S.Ns) return SF3D_INDEX_ERROR;
        set_node_boundary_unchecked(nodeIndex, BT_CULVERT, slope, width * height);
        size_t k = 0;
        for (; k < S.culverts.size(); ++k)
            if (S.culverts[k].roughness == roughness && S.culverts[k].width == width && S.culverts[k].height == height) break;
        if (k == S.culverts.size()) { S.culverts.push_back(CulvertRec{width, height, roughness}); S.tablesDirty = true; }
        S.culvertOf.rw()[nodeIndex] = (uint32_t)k + 1u;         // 0 = no culvert record on this node
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- setNode (soilFluxes3D.cpp:595-629) ---------------------------------------------------------------------
uint8_t sf3d_set_node(uint32_t index, double x, double y, double z, double volume_or_area, int isSurface,
                      uint8_t boundaryType, double slope, double boundaryArea)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(index);
        S.x.rw()[index] = x; S.y.rw()[index] = y; S.z.rw()[index] = z; S.size.rw()[index] = volume_or_area;
        uint32_t *meta = S.meta.rw();
        meta[index] = (meta[index] & ~(1u << 4)) | ((isSurface ? 1u : 0u) << 4);
        set_node_boundary_unchecked(index, boundaryType, slope, boundaryArea);
        if (S.water)
        {
            if (isSurface && index < S.Ns) S.pond.rw()[index] = (double)0.0001f;     // :616 (float literal)
            S.sink.rw()[index] = 0.;
        }
        if (S.heat && !isSurface)                 // soilFluxes3D.cpp:620-626
        {
            S.T.rw()[index] = 273.15 + 20; S.oldT.rw()[index] = 273.15 + 20;
            S.hSink.rw()[index] = 0.;               // heatFlux is device-only and rebuilt every heat sub-step
        }
        S.topoDirty = true;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- setNodeLink (soilFluxes3D.cpp:636-683) -------------------------------------------------------------------
uint8_t sf3d_set_node_link(uint32_t nodeIndex, uint32_t linkIndex, uint8_t direction, double interfaceArea)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (nodeIndex >= S.N || linkIndex >= S.N) return SF3D_INDEX_ERROR;
        uint32_t *meta = S.meta.rw();
        uint32_t m = meta[nodeIndex];
        uint32_t slot;
        switch (direction)
        {
            case 1: slot = 0; break;                 // Up
            case 2: slot = 1; break;                 // Down
            case 3:                                  // Lateral
            {
                const uint32_t nLat = META_NLAT(m);
                if (nLat == SF3D_MAX_LATERAL_LINK) return SF3D_TOPOGRAPHY_ERROR;
                slot = 2 + nLat;
                m = (m & ~(0xFu << 5)) | ((nLat + 1) << 5);
                break;
            }
            default: return SF3D_PARAMETER_ERROR;
        }
        m |= (1u << (9 + slot));
        meta[nodeIndex] = m;
        const size_t li = (size_t)slot * S.N + nodeIndex;
        S.lidx.rw()[li] = linkIndex;
        S.larea.rw()[li] = interfaceArea;
        if (S.water) S.lflow.rw()[li] = 0.;
        if (S.heat)                                   // soilFluxes3D.cpp:669-678 (waterFlux/vaporFlux are zero-initialised on the device)
        {
            double *fx = S.lfluxes.rw();
            fx[li] = SF3D_NODATA;
            if (S.hfMode == 2 && S.hfTypesAllocated == 9)
                for (int t = 1; t < 9; ++t) fx[(size_t)t * SF3D_NLINK * S.N + li] = SF3D_NODATA;
        }
        S.topoDirty = true;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- setNodeSoil / setNodeSurface (soilFluxes3D.cpp:734-775) ------------------------------------------------------
uint8_t sf3d_set_node_soil(uint32_t nodeIndex, uint16_t soilIndex, uint16_t horizonIndex)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (is_surface(nodeIndex)) return SF3D_INDEX_ERROR;
        if (soilIndex >= S.soil1D.size() || horizonIndex >= S.soil1D[soilIndex].size()) return SF3D_PARAMETER_ERROR;
        S.tab.rw()[nodeIndex] = S.soil1D[soilIndex][horizonIndex];
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_set_node_surface(uint32_t nodeIndex, uint16_t surfaceIndex)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (surfaceIndex >= S.rough.size()) return SF3D_PARAMETER_ERROR;
        if (!is_surface(nodeIndex)) return SF3D_INDEX_ERROR;
        S.tab.rw()[nodeIndex] = surfaceIndex;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- water setters (soilFluxes3D.cpp:783-945) -----------------------------------------------------------------------
uint8_t sf3d_set_node_pond(uint32_t nodeIndex, double pond)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (!is_surface(nodeIndex) || nodeIndex >= S.Ns) return SF3D_INDEX_ERROR;
        S.pond.rw()[nodeIndex] = pond;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

static void set_head_and_state(uint32_t i, double H, bool fromSe, double Se)
{
    S.H.rw()[i] = H;
    S.oldH.rw()[i] = H;
    if (is_surface(i)) return;
    if (!fromSe) Se = sf3d_node_se(node_soil(i), g_params.wrcModel, H, S.z.ro()[i]);
    S.Se.rw()[i] = Se;
    S.K.rw()[i] = host_node_K(i, Se);
}

uint8_t sf3d_set_node_water_content(uint32_t nodeIndex, double waterContent)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (waterContent < 0.) return SF3D_PARAMETER_ERROR;
        if (is_surface(nodeIndex))
        {
            const double H = S.z.ro()[nodeIndex] + waterContent;
            S.H.rw()[nodeIndex] = H; S.oldH.rw()[nodeIndex] = H;
            S.Se.rw()[nodeIndex] = 1.; S.K.rw()[nodeIndex] = 0.;
        }
        else
        {
            if (waterContent > 1.) return SF3D_PARAMETER_ERROR;
            const SoilRec &s = node_soil(nodeIndex);
            const double Se = host_se_from_theta(s, waterContent);
            set_head_and_state(nodeIndex, S.z.ro()[nodeIndex] - host_psi_from_se(s, Se), true, Se);
        }
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_set_node_degree_of_saturation(uint32_t nodeIndex, double Se)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (is_surface(nodeIndex)) return SF3D_INDEX_ERROR;
        if (Se < 0. || Se > 1.) return SF3D_PARAMETER_ERROR;
        set_head_and_state(nodeIndex, S.z.ro()[nodeIndex] - host_psi_from_se(node_soil(nodeIndex), Se), true, Se);
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
static uint8_t set_potential(uint32_t i, double H)
{
    S.H.rw()[i] = H; S.oldH.rw()[i] = H;
    if (is_surface(i)) { S.Se.rw()[i] = 1.; S.K.rw()[i] = SF3D_NODATA; }
    else set_head_and_state(i, H, false, 0.);
    return SF3D_OK;
}
uint8_t sf3d_set_node_matric_potential(uint32_t nodeIndex, double psi)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        return set_potential(nodeIndex, S.z.ro()[nodeIndex] + psi);
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_set_node_total_potential(uint32_t nodeIndex, double H)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        return set_potential(nodeIndex, H);
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_set_node_water_sink_source(uint32_t nodeIndex, double q)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        S.sink.rw()[nodeIndex] = q;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_set_node_prescribed_total_potential(uint32_t nodeIndex, double H)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(nodeIndex);
        if (node_bt(nodeIndex) != BT_PRESCRIBED) return SF3D_BOUNDARY_ERROR;
        S.bPresc.rw()[nodeIndex] = H;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- water getters (soilFluxes3D.cpp:951-1277) ---------------------------------------------------------------------------
#define GETTER_PROLOGUE(i) REQUIRE_INIT_D(); REQUIRE_INDEX_D(i)
#define GUARDED_D(...) return guarded([&]() -> double { __VA_ARGS__ }, err_value(SF3D_MEMORY_ERROR))

double sf3d_get_node_water_content(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i);
    return is_surface(i) ? (S.H.ro()[i] - S.z.ro()[i]) : sf3d_theta_from_se(node_soil(i), S.Se.ro()[i]); ); }
double sf3d_get_node_maximum_water_content(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (is_surface(i)) return err_value(SF3D_INDEX_ERROR); return node_soil(i).thetaS; ); }
double sf3d_get_node_minimum_water_content(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (is_surface(i)) return err_value(SF3D_INDEX_ERROR); return node_soil(i).thetaR; ); }
double sf3d_get_node_available_water_content(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i);
    if (is_surface(i)) return S.H.ro()[i] - S.z.ro()[i];
    const SoilRec &s = node_soil(i);
    return sf3d_max(0., sf3d_theta_from_se(s, S.Se.ro()[i]) - sf3d_theta_from_signed_psi(s, g_params.wrcModel, -160)); ); }
double sf3d_get_node_water_deficit(uint32_t i, double fieldCapacity)
{ GUARDED_D( GETTER_PROLOGUE(i);
    if (is_surface(i)) return 0.;
    const SoilRec &s = node_soil(i);
    return sf3d_theta_from_signed_psi(s, g_params.wrcModel, -fieldCapacity) - sf3d_theta_from_se(s, S.Se.ro()[i]); ); }
double sf3d_get_node_degree_of_saturation(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i);
    if (!is_surface(i)) return S.Se.ro()[i];
    const double curPot = S.H.ro()[i] - S.z.ro()[i], maxPot = 0.001;
    return curPot <= 0 ? 0 : (curPot > maxPot ? 1. : curPot / maxPot); ); }
double sf3d_get_node_water_conductivity(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return S.K.ro()[i]; ); }
double sf3d_get_node_matric_potential(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return S.H.ro()[i] - S.z.ro()[i]; ); }
double sf3d_get_node_total_potential(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return S.H.ro()[i]; ); }
double sf3d_get_node_pond(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (!is_surface(i) || i >= S.Ns) return err_value(SF3D_INDEX_ERROR); return S.pond.ro()[i]; ); }

double sf3d_get_node_max_water_flow(uint32_t i, uint8_t direction)
{ GUARDED_D( GETTER_PROLOGUE(i);
    const double *lf = S.lflow.ro();
    const uint32_t m = S.meta.ro()[i];
    switch (direction)
    {
        case 1: return lf[i];                       // linkIndex is calloc'ed, never noDataU: always the stored sum
        case 2: return lf[(size_t)S.N + i];
        case 3:
        {
            double mx = 0.;
            for (uint32_t l = 0; l < META_NLAT(m); ++l) mx = sf3d_max(mx, lf[(size_t)(2 + l) * S.N + i]);
            return mx;
        }
        default: return err_value(SF3D_INDEX_ERROR);
    } ); }
static double lateral_sum(uint32_t i, int sign)
{
    const double *lf = S.lflow.ro();
    const uint32_t m = S.meta.ro()[i];
    double sum = 0.;
    for (uint32_t l = 0; l < META_NLAT(m); ++l)
    {
        const double f = lf[(size_t)(2 + l) * S.N + i];
        if (sign == 0 || (sign > 0 && f > 0) || (sign < 0 && f < 0)) sum += f;
    }
    return sum;
}
double sf3d_get_node_sum_lateral_water_flow(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return lateral_sum(i, 0); ); }
double sf3d_get_node_sum_lateral_water_flow_in(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return lateral_sum(i, 1); ); }
double sf3d_get_node_sum_lateral_water_flow_out(uint32_t i) { GUARDED_D( GETTER_PROLOGUE(i); return lateral_sum(i, -1); ); }
double sf3d_get_node_boundary_water_flow(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (node_bt(i) == BT_NONE) return err_value(SF3D_BOUNDARY_ERROR); return S.bSum.ro()[i]; ); }

double sf3d_get_total_boundary_water_flow(uint8_t boundaryType)
{ GUARDED_D(
    if (!S.initialized) return 0.;
    if (sync_to_device()) return 0.;
    return S.eng.totalBoundaryWaterFlow(boundaryType); ); }
double sf3d_get_total_water_content(void)
{ GUARDED_D(
    if (!S.initialized) return -1;                  // water.cpp:73-74
    if (sync_to_device()) return -1;
    return S.eng.totalWaterContent(); ); }
double sf3d_get_water_storage(void) { return S.eng.curStep.waterStorage; }
double sf3d_get_water_mbr(void) { return S.eng.wholePeriod.waterMBR; }

// ---- heat API (soilFluxes3D.cpp:1283-1753) ---------------------------------------------------------------------------------
#define REQUIRE_HEAT_E() do { if (!S.heat) return SF3D_MISSING_DATA_ERROR; } while (0)   /* the reference would touch null arrays */
static SF3DView host_view()
{
    // a view over the HOST mirrors for the getters that evaluate closures on one node
    SF3DView v = S.eng.v;
    v.z = const_cast<double *>(S.z.ro()); v.size = const_cast<double *>(S.size.ro());
    v.tab = const_cast<uint16_t *>(S.tab.ro()); v.meta = const_cast<uint32_t *>(S.meta.ro());
    v.H = const_cast<double *>(S.H.ro()); v.oldH = const_cast<double *>(S.oldH.ro());
    v.T = const_cast<double *>(S.T.ro()); v.oldT = const_cast<double *>(S.oldT.ro());
    v.soil = S.soils.data();
    v.wrcModel = g_params.wrcModel;
    v.computeHeatVapor = S.heatVapor;
    v.hPress = nullptr; v.ldist3 = nullptr; v.hTm = v.hTLK = v.hTLKh = nullptr; v.hHs = v.hPsiAvg = v.hInv = nullptr;      // device-only tables
    return v;
}
uint8_t sf3d_set_node_heat_sink_source(uint32_t i, double q)
{ return guarded([&]() -> uint8_t { REQUIRE_INIT_E(); REQUIRE_INDEX_E(i); REQUIRE_HEAT_E(); S.hSink.rw()[i] = q; return SF3D_OK; }, (uint8_t)SF3D_MEMORY_ERROR); }
uint8_t sf3d_set_node_temperature(uint32_t i, double T)
{ return guarded([&]() -> uint8_t { REQUIRE_INIT_E(); REQUIRE_INDEX_E(i); REQUIRE_HEAT_E(); S.T.rw()[i] = T; S.oldT.rw()[i] = T; return SF3D_OK; }, (uint8_t)SF3D_MEMORY_ERROR); }
uint8_t sf3d_set_node_boundary_fixed_temperature(uint32_t i, double T, double depth)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E(); REQUIRE_INDEX_E(i); REQUIRE_HEAT_E();
        const uint32_t bt = node_bt(i);
        if (bt != BT_PRESCRIBED && bt != BT_FREE_DRAINAGE) return SF3D_BOUNDARY_ERROR;
        S.hbFixT.rw()[i] = T; S.hbFixDepth.rw()[i] = depth;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
#define HEAT_BOUNDARY_SETTER(name, mirror, extraCheck)                                              \
    uint8_t name(uint32_t i, double value)                                                         \
    {                                                                                              \
        return guarded([&]() -> uint8_t {                                                          \
            REQUIRE_INIT_E(); REQUIRE_INDEX_E(i); REQUIRE_HEAT_E();                                \
            if (node_bt(i) == BT_NONE) return SF3D_BOUNDARY_ERROR;                                 \
            extraCheck                                                                             \
            S.mirror.rw()[i] = value;                                                              \
            return SF3D_OK;                                                                        \
        }, (uint8_t)SF3D_MEMORY_ERROR);                                                            \
    }
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_height_wind, hbHeightWind, )
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_height_temperature, hbHeightT, )
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_net_irradiance, hbNetIrr, )
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_temperature, hbT, )
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_relative_humidity, hbRH, )
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_roughness, hbRough, if (value < 0) return SF3D_PARAMETER_ERROR;)
HEAT_BOUNDARY_SETTER(sf3d_set_node_boundary_wind_speed, hbWind, if ((value < 0.) || (value > 1000.)) return SF3D_PARAMETER_ERROR;)

static bool is_heat_node(uint32_t i) { return S.heat && !is_surface(i); }       // heat.cpp:26-29
double sf3d_get_node_temperature(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (!is_heat_node(i)) return err_value(SF3D_TOPOGRAPHY_ERROR); return S.T.ro()[i]; ); }
double sf3d_get_node_heat_conductivity(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i); if (!is_heat_node(i)) return err_value(SF3D_TOPOGRAPHY_ERROR);
    const SF3DView hv = host_view();
    return h_soil_heat_conductivity(hv, i, hv.T[i], hv.H[i] - hv.z[i]); ); }
double sf3d_get_node_vapor(uint32_t i)
{ GUARDED_D( GETTER_PROLOGUE(i);
    if (!S.water || !S.heat || !S.heatVapor) return err_value(SF3D_MISSING_DATA_ERROR);
    return h_vapor_from_psi_temp(S.H.ro()[i] - S.z.ro()[i], S.T.ro()[i]); ); }
double sf3d_get_node_heat_storage(uint32_t i, double h)
{ GUARDED_D( GETTER_PROLOGUE(i); if (!S.heat) return err_value(SF3D_MISSING_DATA_ERROR);
    const SF3DView hv = host_view();
    return h_node_heat_storage(hv, i, h); ); }
static double link_heat_flux(uint32_t slot, uint32_t i, uint8_t fluxType)        // getLinkHeatFlux, heat.cpp:623-641
{
    if (!S.heat) return SF3D_NODATA;
    if (S.hfMode == 1) return (fluxType == 0) ? S.lfluxes.ro()[(size_t)slot * S.N + i] : SF3D_NODATA;
    if (S.hfMode == 2 && S.hfTypesAllocated == 9) return S.lfluxes.ro()[((size_t)fluxType * SF3D_NLINK + slot) * S.N + i];
    return SF3D_NODATA;
}
double sf3d_get_node_heat_max_flux(uint32_t i, uint8_t direction, uint8_t fluxType)
{ GUARDED_D( GETTER_PROLOGUE(i); if (!is_heat_node(i)) return err_value(SF3D_TOPOGRAPHY_ERROR);
    if (fluxType > 8) return err_value(SF3D_INDEX_ERROR);
    switch (direction)
    {
        case 1: return link_heat_flux(0, i, fluxType);
        case 2: return link_heat_flux(1, i, fluxType);
        case 3:
        {
            double mx = 0.;
            for (uint32_t l = 0; l < SF3D_MAX_LATERAL_LINK; ++l)
            {
                const double f = link_heat_flux(2 + l, i, fluxType);
                if (f > fabs(mx)) mx = f;
            }
            return mx;
        }
        default: return err_value(SF3D_INDEX_ERROR);
    } ); }
#define HEAT_BOUNDARY_GETTER(name, mirror, needVapor)                                               \
    double name(uint32_t i)                                                                        \
    { GUARDED_D( GETTER_PROLOGUE(i);                                                                \
        if (needVapor ? (!S.water || !S.heat || !S.heatVapor) : !S.heat) return err_value(SF3D_MISSING_DATA_ERROR); \
        if (node_bt(i) != BT_HEAT_SURFACE) return err_value(SF3D_BOUNDARY_ERROR);                  \
        return S.mirror.ro()[i]; ); }
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_advective_flux, hbAdv, true)
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_latent_flux, hbLat, true)
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_radiative_flux, hbRad, false)
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_sensible_flux, hbSens, false)
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_aerodynamic_conductance, hbAero, false)
HEAT_BOUNDARY_GETTER(sf3d_get_node_boundary_soil_conductance, hbSoilCond, false)
double sf3d_get_heat_mbr(void) { return S.eng.wholePeriod.heatMBR; }
double sf3d_get_heat_mbe(void) { return S.eng.wholePeriod.heatMBE; }

// ---- computation (soilFluxes3D.cpp:1760-1821) ----------------------------------------------------------------------------------
double sf3d_compute_step(double maxTimeStep)
{
    g_lastStepError = SF3D_OK;
    return guarded([&]() -> double {
        if (!S.initialized) return err_value(SF3D_MEMORY_ERROR);
        if (sync_to_device()) return err_value(SF3D_TOPOGRAPHY_ERROR);
        const double dt = S.eng.computeStep(maxTimeStep);
        step_wrote_device();
        return dt;
    }, err_value(SF3D_MEMORY_ERROR));
}
void sf3d_compute_period(double timePeriod)
{
    g_lastStepError = SF3D_OK;
    guarded([&]() -> int {
        if (!S.initialized) return 0;
        if (sync_to_device()) return 0;
        S.eng.computePeriod(timePeriod);
        step_wrote_device();
        return 0;
    }, 0);
}

// ====================================== extensions ===================================================
uint8_t sf3d_ext_get_field(int field, uint32_t first, uint32_t count, double *dst)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!dst) return SF3D_PARAMETER_ERROR;
        if ((uint64_t)first + count > S.N) return SF3D_INDEX_ERROR;
        switch (field)
        {
            case SF3D_F_WATER_CONTENT: case SF3D_F_DEGREE_OF_SATURATION: case SF3D_F_WATER_CONDUCTIVITY:
            case SF3D_F_MATRIC_POTENTIAL: case SF3D_F_TOTAL_POTENTIAL: case SF3D_F_POND:
            case SF3D_F_BOUNDARY_WATER_FLOW: case SF3D_F_SUM_LATERAL_FLOW: case SF3D_F_MAX_FLOW_UP:
            case SF3D_F_MAX_FLOW_DOWN: case SF3D_F_MAX_FLOW_LATERAL: case SF3D_F_TEMPERATURE:
                break;
            default: return SF3D_PARAMETER_ERROR;
        }
        uint8_t rc = sync_to_device();
        if (rc) return rc;
        if (field == SF3D_F_TOTAL_POTENTIAL)        // getNodeTotalPotential is the array itself: one copy
        {
            d2h(dst, S.H.d + first, (size_t)count * sizeof(double));
            return SF3D_OK;
        }
        double *tmp = scratch_buffer();
        k_get_field(S.eng.v, field, first, count, tmp);
        d2h(dst, tmp, (size_t)count * sizeof(double));
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

uint8_t sf3d_ext_set_field(int field, uint32_t first, uint32_t count, const double *src)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!src) return SF3D_PARAMETER_ERROR;
        if ((uint64_t)first + count > S.N) return SF3D_INDEX_ERROR;
        switch (field)
        {
            case SF3D_F_WATER_SINK_SOURCE:          // setNodeWaterSinkSource over a range: one copy
                S.sink.push();
                h2d(S.sink.d + first, src, (size_t)count * sizeof(double));
                S.sink.dev_written();
                return SF3D_OK;
            case SF3D_F_MATRIC_POTENTIAL: case SF3D_F_TOTAL_POTENTIAL:
            {
                uint8_t rc = sync_to_device();
                if (rc) return rc;
                double *tmp = scratch_buffer();
                h2d(tmp, src, (size_t)count * sizeof(double));
                k_set_potential(S.eng.v, first, count, tmp, field == SF3D_F_TOTAL_POTENTIAL);
                S.eng.tryPrepared = false;
                S.H.dev_written(); S.oldH.dev_written(); S.Se.dev_written(); S.K.dev_written();
                return SF3D_OK;
            }
            default: break;
        }
        // remaining fields: the scalar setter per node on the host mirrors
        uint8_t firstErr = SF3D_OK;
        for (uint32_t k = 0; k < count; ++k)
        {
            const uint32_t i = first + k;
            uint8_t rc;
            switch (field)
            {
                case SF3D_F_WATER_CONTENT:        rc = sf3d_set_node_water_content(i, src[k]); break;
                case SF3D_F_DEGREE_OF_SATURATION: rc = sf3d_set_node_degree_of_saturation(i, src[k]); break;
                case SF3D_F_POND:                 rc = sf3d_set_node_pond(i, src[k]); break;
                case SF3D_F_PRESCRIBED_POTENTIAL: rc = sf3d_set_node_prescribed_total_potential(i, src[k]); break;
                case SF3D_F_TEMPERATURE:          rc = sf3d_set_node_temperature(i, src[k]); break;
                case SF3D_F_HEAT_SINK_SOURCE:     rc = sf3d_set_node_heat_sink_source(i, src[k]); break;
                case SF3D_F_BOUNDARY_NET_IRRADIANCE:    rc = sf3d_set_node_boundary_net_irradiance(i, src[k]); break;
                case SF3D_F_BOUNDARY_TEMPERATURE:       rc = sf3d_set_node_boundary_temperature(i, src[k]); break;
                case SF3D_F_BOUNDARY_RELATIVE_HUMIDITY: rc = sf3d_set_node_boundary_relative_humidity(i, src[k]); break;
                case SF3D_F_BOUNDARY_WIND_SPEED:        rc = sf3d_set_node_boundary_wind_speed(i, src[k]); break;
                case SF3D_F_BOUNDARY_HEIGHT_WIND:       rc = sf3d_set_node_boundary_height_wind(i, src[k]); break;
                case SF3D_F_BOUNDARY_HEIGHT_TEMPERATURE: rc = sf3d_set_node_boundary_height_temperature(i, src[k]); break;
                case SF3D_F_BOUNDARY_ROUGHNESS:         rc = sf3d_set_node_boundary_roughness(i, src[k]); break;
                default: return SF3D_PARAMETER_ERROR;
            }
            if (rc && !firstErr) firstErr = rc;
        }
        return firstErr;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

uint8_t sf3d_ext_get_link_table(uint8_t slot, uint32_t first, uint32_t count, uint8_t *lt, uint32_t *li, double *area)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (slot >= SF3D_NLINK || (uint64_t)first + count > S.N) return SF3D_INDEX_ERROR;
        const uint32_t *meta = S.meta.ro();
        const uint32_t *lidx = S.lidx.ro();
        const double *larea = S.larea.ro();
        for (uint32_t k = 0; k < count; ++k)
        {
            const uint32_t i = first + k;
            const bool has = META_HAS_SLOT(meta[i], slot);
            if (lt) lt[k] = has ? (slot == 0 ? 1 : (slot == 1 ? 2 : 3)) : 0;
            if (li) li[k] = has ? lidx[(size_t)slot * S.N + i] : 0u;
            if (area) area[k] = has ? larea[(size_t)slot * S.N + i] : 0.;
        }
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

uint8_t sf3d_ext_get_node_meta(uint32_t first, uint32_t count, uint8_t *sfl, uint8_t *bt, uint8_t *nl)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if ((uint64_t)first + count > S.N) return SF3D_INDEX_ERROR;
        const uint32_t *meta = S.meta.ro();
        for (uint32_t k = 0; k < count; ++k)
        {
            const uint32_t m = meta[first + k];
            if (sfl) sfl[k] = (uint8_t)META_SURFACE(m);
            if (bt) bt[k] = (uint8_t)META_BT(m);
            if (nl) nl[k] = (uint8_t)META_NLAT(m);
        }
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

uint8_t sf3d_ext_build_grid(const sf3d_grid_desc *g)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!g || !g->dem || !g->cell_rank || !g->layer_depth || !g->layer_thickness) return SF3D_PARAMETER_ERROR;
        const uint64_t cells = (uint64_t)g->rows * g->cols;
        if ((uint64_t)g->layers * g->n_valid != S.N || g->n_valid != S.Ns) return SF3D_INDEX_ERROR;

        // soil-table row of every (soil id, layer) pair; setNodeSoil's checks (soilFluxes3D.cpp:745-746)
        uint32_t nSoilIds = 1;
        if (g->soil_id) for (uint64_t c = 0; c < cells; ++c) if (g->cell_rank[c] >= 0) nSoilIds = std::max<uint32_t>(nSoilIds, g->soil_id[c] + 1u);
        std::vector<uint16_t> layerTab((size_t)g->layers * nSoilIds, 0);
        std::vector<uint8_t> used(nSoilIds, g->soil_id ? 0 : 1);
        if (g->soil_id) for (uint64_t c = 0; c < cells; ++c) if (g->cell_rank[c] >= 0) used[g->soil_id[c]] = 1;
        for (uint32_t l = 1; l < g->layers; ++l)
            for (uint32_t sid = 0; sid < nSoilIds; ++sid)
            {
                if (!used[sid]) continue;
                const uint16_t hz = g->layer_horizon ? g->layer_horizon[l] : 0;
                if (sid >= S.soil1D.size() || hz >= S.soil1D[sid].size()) return SF3D_PARAMETER_ERROR;
                layerTab[(size_t)l * nSoilIds + sid] = S.soil1D[sid][hz];
            }
        if (g->surface_id) for (uint64_t c = 0; c < cells; ++c)
            if (g->cell_rank[c] >= 0 && g->surface_id[c] >= S.rough.size()) return SF3D_PARAMETER_ERROR;

        uint8_t rc = sync_to_device(false);     // pushes anything set so far; view is current
        if (rc) return rc;

        std::vector<void *> tmp;
        auto up = [&](const void *src, size_t bytes) -> void * {
            if (!src) return nullptr;
            void *d = dev_alloc(bytes); h2d(d, src, bytes); tmp.push_back(d); return d;
        };
        GridDev gd{};
        gd.rows = g->rows; gd.cols = g->cols; gd.layers = g->layers; gd.nValid = g->n_valid;
        gd.cell = g->cell; gd.xll = g->x_ll; gd.yll = g->y_ll;
        gd.dem = (const float *)up(g->dem, cells * 4);
        gd.slope = (const float *)up(g->slope_tan, cells * 4);
        gd.rank = (const int32_t *)up(g->cell_rank, cells * 4);
        gd.outlet = (const uint8_t *)up(g->outlet, cells);
        gd.boundaryL1 = (const uint8_t *)up(g->boundary_l1, cells);
        gd.soilId = (const uint16_t *)up(g->soil_id, cells * 2);
        gd.surfaceId = (const uint16_t *)up(g->surface_id, cells * 2);
        gd.pond = (const double *)up(g->pond, cells * 8);
        gd.layerDepth = (const double *)up(g->layer_depth, (size_t)g->layers * 8);
        gd.layerThickness = (const double *)up(g->layer_thickness, (size_t)g->layers * 8);
        gd.layerTab = (const uint16_t *)up(layerTab.data(), layerTab.size() * 2);
        gd.nSoilIds = nSoilIds;
        gd.freeRunoff = g->free_catchment_runoff; gd.freeLateral = g->free_lateral_drainage; gd.freeBottom = g->free_bottom_drainage;
        gd.computeWater = S.water; gd.computeHeat = S.heat; gd.heatSurfaceL1 = g->heat_surface_layer1;
        k_build_grid(S.eng.v, gd);
        dev_sync();
        // the cell -> node map stays on the device for sf3d_ext_set_forcing_rasters / sf3d_ext_get_layer_raster
        dev_free(S.rasterRank); S.rasterRank = nullptr;
        for (void *&d : tmp) if (d == (void *)gd.rank) { S.rasterRank = (int32_t *)d; d = nullptr; }
        S.raster.rows = g->rows; S.raster.cols = g->cols; S.raster.layers = g->layers; S.raster.nValid = g->n_valid;
        S.raster.cell = g->cell; S.raster.rank = S.rasterRank;
        for (void *d : tmp) dev_free(d);

        S.x.dev_written(); S.y.dev_written(); S.z.dev_written(); S.size.dev_written(); S.meta.dev_written();
        S.tab.dev_written(); S.bSlope.dev_written(); S.bSize.dev_written(); S.bRate.dev_written();
        S.bSum.dev_written(); S.bPresc.dev_written(); S.lidx.dev_written(); S.larea.dev_written();
        S.sink.dev_written(); S.pond.dev_written();
        if (S.heat)
        {
            S.T.dev_written(); S.oldT.dev_written(); S.hSink.dev_written(); S.lfluxes.dev_written();
            collect_heat_mirrors();
            for (Mirror<double> *m : heat_boundary_mirrors) m->dev_written();
        }
        S.topoDirty = true;
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

// ---- raster-facing forcing / output (SURVEY 8 f3, f4; semantics in include/sf3d.h) ----------------
uint8_t sf3d_ext_set_forcing_rasters(const sf3d_forcing_desc *f)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!f) return SF3D_PARAMETER_ERROR;
        if (!S.rasterRank) return SF3D_MISSING_DATA_ERROR;
        if (f->rows != S.raster.rows || f->cols != S.raster.cols) return SF3D_PARAMETER_ERROR;
        if (f->layer_sink && f->n_sink_layers > S.raster.layers) return SF3D_PARAMETER_ERROR;
        uint8_t rc = sync_to_device();
        if (rc) return rc;
        const size_t cells = (size_t)f->rows * f->cols;
        const size_t nPrec = f->precipitation ? cells : 0, nSink = f->layer_sink ? cells * f->n_sink_layers : 0;
        float *stage = (float *)raster_stage((nPrec + nSink + 1) * sizeof(float));
        ForcingDev fd{};
        if (nPrec) { h2d(stage, f->precipitation, nPrec * sizeof(float)); fd.precipitation = stage; }
        if (nSink) { h2d(stage + nPrec, f->layer_sink, nSink * sizeof(float)); fd.layerSink = stage + nPrec; }
        fd.precipitationNodata = f->precipitation_nodata; fd.sinkNodata = f->sink_nodata;
        fd.nSinkLayers = f->n_sink_layers; fd.accumulate = f->accumulate;
        S.sink.push();
        k_forcing_rasters(S.eng.v, S.raster, fd);
        S.sink.dev_written();
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}

static uint8_t layer_rasters(int field, uint32_t firstLayer, uint32_t nLayers, float nodata, float *dst, bool overlapped)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!dst) return SF3D_PARAMETER_ERROR;
        if (!S.rasterRank) return SF3D_MISSING_DATA_ERROR;
        if ((uint64_t)firstLayer + nLayers > S.raster.layers || nLayers == 0) return SF3D_INDEX_ERROR;
        switch (field)
        {
            case SF3D_F_WATER_CONTENT: case SF3D_F_DEGREE_OF_SATURATION: case SF3D_F_WATER_CONDUCTIVITY:
            case SF3D_F_MATRIC_POTENTIAL: case SF3D_F_TOTAL_POTENTIAL: case SF3D_F_POND:
            case SF3D_F_BOUNDARY_WATER_FLOW: case SF3D_F_SUM_LATERAL_FLOW: case SF3D_F_MAX_FLOW_UP:
            case SF3D_F_MAX_FLOW_DOWN: case SF3D_F_MAX_FLOW_LATERAL: case SF3D_F_TEMPERATURE:
                break;
            default: return SF3D_PARAMETER_ERROR;
        }
        uint8_t rc = sync_to_device();
        if (rc) return rc;
        const size_t cells = (size_t)S.raster.rows * S.raster.cols, bytes = cells * nLayers * sizeof(float);
        float *stage;
        int slot = 0;
        if (overlapped)
        {
            // two staging buffers of their own (the forcing upload uses the shared one): a copy may still be reading one of
            // them while the next maps are written into the other
            slot = S.overlapSlot ^= 1;
            if (S.overlapStageBytes[slot] < bytes)
            {
                overlap_sync();
                dev_free(S.overlapStage[slot]); S.overlapStage[slot] = nullptr; S.overlapStageBytes[slot] = 0;
                S.overlapStage[slot] = dev_alloc(bytes); S.overlapStageBytes[slot] = bytes;
            }
            overlap_acquire(slot);
            stage = (float *)S.overlapStage[slot];
        }
        else stage = (float *)raster_stage(bytes);
        for (uint32_t l = 0; l < nLayers; ++l) k_layer_raster(S.eng.v, S.raster, field, firstLayer + l, nodata, stage + (size_t)l * cells);
        if (overlapped) d2h_overlapped(dst, stage, bytes, slot);
        else d2h(dst, stage, bytes);
        return SF3D_OK;
    }, (uint8_t)SF3D_MEMORY_ERROR);
}
uint8_t sf3d_ext_get_layer_rasters(int field, uint32_t firstLayer, uint32_t nLayers, float nodata, float *dst)
{ return layer_rasters(field, firstLayer, nLayers, nodata, dst, false); }
uint8_t sf3d_ext_get_layer_rasters_async(int field, uint32_t firstLayer, uint32_t nLayers, float nodata, float *dst)
{ return layer_rasters(field, firstLayer, nLayers, nodata, dst, true); }
uint8_t sf3d_ext_wait_rasters(void)
{ return guarded([&]() -> uint8_t { overlap_sync(); return SF3D_OK; }, (uint8_t)SF3D_MEMORY_ERROR); }

uint8_t sf3d_ext_set_fixed_temperature(uint32_t first, uint32_t count, const double *temperature, double depth)
{
    if (!temperature) return SF3D_PARAMETER_ERROR;
    uint8_t firstErr = SF3D_OK;
    for (uint32_t k = 0; k < count; ++k)
    {
        uint8_t rc = sf3d_set_node_boundary_fixed_temperature(first + k, temperature[k], depth);
        if (rc && !firstErr) firstErr = rc;
    }
    return firstErr;
}

uint8_t sf3d_ext_get_counters(sf3d_counters *out)
{
    if (!out) return SF3D_PARAMETER_ERROR;
    sf3d_counters c = S.eng.cnt;
    c.kernel_launches = launches();
    c.delta_t_curr = g_params.deltaTcurr;
    c.last_courant = S.eng.courantWater;
    c.last_mbr = S.eng.curStep.waterMBR;
    c.last_mbe = S.eng.curStep.waterMBE;
    c.links = 0;
    if (S.initialized)
        c.links = guarded([&]() -> uint64_t { if (sync_to_device(false)) return 0; return k_count_links(S.eng.v); }, (uint64_t)0);
    *out = c;
    return SF3D_OK;
}
uint8_t sf3d_ext_reset_counters(void) { memset(&S.eng.cnt, 0, sizeof S.eng.cnt); return SF3D_OK; }
uint8_t sf3d_ext_last_error(void) { const uint8_t e = g_lastStepError; g_lastStepError = SF3D_OK; return e; }
const char *sf3d_ext_backend(void) { return "b200"; }
uint8_t sf3d_ext_set_device(int device)
{
    if (S.initialized) return SF3D_PARAMETER_ERROR;     // choose the device before initializeSF3D
    g_device = device;
    return SF3D_OK;
}

uint8_t sf3d_ext_reset_solver(void) { g_params = default_params(); return SF3D_OK; }
uint8_t sf3d_ext_set_time_step(double deltaT) { g_params.deltaTcurr = deltaT; return SF3D_OK; }     // solver.h:77-86

uint8_t sf3d_ext_jacobi_sweep(uint32_t n, uint32_t nSurface, const uint8_t *ncols, const uint32_t *col, const double *val,
                              const double *b, const double *z, const double *xIn, double *xOut, double *norm)
{
    if (!ncols || !col || !val || !b || !z || !xIn || !xOut || !norm || n == 0) return SF3D_PARAMETER_ERROR;
    return guarded([&]() -> uint8_t {
        dev_select(g_device);
        // compact rows -> the product's fixed ten-column layout, column order preserved; absent entries 0 / self
        std::vector<double> mv((size_t)SF3D_NLINK * n, 0.0);
        std::vector<uint32_t> mc((size_t)SF3D_NLINK * n);
        for (uint32_t r = 0; r < n; ++r)
            for (int c = 0; c < SF3D_NLINK; ++c)
            {
                const bool has = (c + 1) < ncols[r];
                mv[(size_t)c * n + r] = has ? val[(size_t)r * 11 + c + 1] : 0.0;
                mc[(size_t)c * n + r] = has ? col[(size_t)r * 11 + c + 1] : r;
            }
        SF3DView v{};
        v.N = n; v.Ns = nSurface; v.world = 1; v.nGlobal = (double)n;
        double *dmv = (double *)dev_alloc(mv.size() * 8); uint32_t *dmc = (uint32_t *)dev_alloc(mc.size() * 4);
        double *db = (double *)dev_alloc((size_t)n * 8), *dz = (double *)dev_alloc((size_t)n * 8);
        double *dx0 = (double *)dev_alloc((size_t)n * 8), *dx1 = (double *)dev_alloc((size_t)n * 8);
        const size_t nb = (size_t)std::max(reduce_blocks(0xFFFFFFFFu), wide_blocks(0xFFFFFFFFu));
        double *part = (double *)dev_alloc(nb * 8);
        Ctrl *ctrl = (Ctrl *)dev_alloc(sizeof(Ctrl));
        h2d(dmv, mv.data(), mv.size() * 8); h2d(dmc, mc.data(), mc.size() * 4);
        h2d(db, b, (size_t)n * 8); h2d(dz, z, (size_t)n * 8); h2d(dx0, xIn, (size_t)n * 8);
        v.mval = dmv; v.mcol = dmc; v.b = db; v.z = dz; v.ctrl = ctrl; v.partA = part; v.pid = nullptr; v.pattern = nullptr;
        Ctrl c0{}; c0.status = SOLVE_RUNNING; c0.bestNorm = 1.;
        write_ctrl(v, &c0);
        k_jacobi(v, dx0, dx1, 1000000, 0.0);
        Ctrl c1{};
        read_ctrl(v, &c1);
        d2h(xOut, dx1, (size_t)n * 8);
        *norm = c1.lastNorm;
        for (void *p : {(void *)dmv, (void *)dmc, (void *)db, (void *)dz, (void *)dx0, (void *)dx1, (void *)part, (void *)ctrl}) dev_free(p);
        return SF3D_OK;
    }, (uint8_t)SF3D_SOLVER_ERROR);
}

uint8_t sf3d_ext_comm_unique_id(uint8_t id[128])
{ return guarded([&]() -> uint8_t { dev_select(g_device); comm_unique_id(id); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR); }
uint8_t sf3d_ext_comm_init(int rank, int world, const uint8_t id[128])
{
    if (S.initialized) return SF3D_PARAMETER_ERROR;     // wire the ranks before initializeSF3D
    // id == NULL: peer memory only, no NCCL communicator (see comm_init)
    return guarded([&]() -> uint8_t { dev_select(g_device); comm_init(rank, world, id); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR);
}
uint8_t sf3d_ext_ipc_export(uint8_t handles[128])
{
    return guarded([&]() -> uint8_t { REQUIRE_INIT_E(); comm_ipc_export(S.x0, S.x1, handles); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR);
}
uint8_t sf3d_ext_ipc_import(int peer, const uint8_t handles[128], uint32_t n, const uint32_t *remoteIdx)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (!handles || (n && !remoteIdx)) return SF3D_PARAMETER_ERROR;
        comm_ipc_import(peer, handles, n, remoteIdx);
        return SF3D_OK;
    }, (uint8_t)SF3D_SOLVER_ERROR);
}
uint8_t sf3d_ext_mailbox_export(uint8_t handle[64])
{ return guarded([&]() -> uint8_t { dev_select(g_device); comm_mailbox_export(handle); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR); }
uint8_t sf3d_ext_mailbox_import(int peer, const uint8_t handle[64])
{
    if (!handle) return SF3D_PARAMETER_ERROR;
    return guarded([&]() -> uint8_t { comm_mailbox_import(peer, handle); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR);
}
uint8_t sf3d_ext_comm_finalize(void)
{ return guarded([&]() -> uint8_t { comm_finalize(); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR); }
uint8_t sf3d_ext_set_halo(uint32_t nPeers, const int32_t *peers, const uint32_t *sendCount, const uint32_t *sendIdx,
                          const uint32_t *recvCount, const uint32_t *recvIdx, uint64_t nGlobalNodes)
{
    return guarded([&]() -> uint8_t {
        REQUIRE_INIT_E();
        if (nPeers && (!peers || !sendCount || !recvCount)) return SF3D_PARAMETER_ERROR;
        comm_clear_halo();
        uint32_t *meta = S.meta.rw();
        for (uint32_t i = 0; i < S.N; ++i) meta[i] &= ~(1u << 19);
        size_t so = 0, ro = 0;
        for (uint32_t p = 0; p < nPeers; ++p)
        {
            for (uint32_t k = 0; k < sendCount[p]; ++k) if (sendIdx[so + k] >= S.N) return SF3D_INDEX_ERROR;
            for (uint32_t k = 0; k < recvCount[p]; ++k)
            {
                if (recvIdx[ro + k] >= S.N) return SF3D_INDEX_ERROR;
                meta[recvIdx[ro + k]] |= (1u << 19);               // ghost
            }
            comm_add_halo_peer(peers[p], sendCount[p], sendIdx + so, recvCount[p], recvIdx + ro);
            so += sendCount[p]; ro += recvCount[p];
        }
        S.nGlobal = (double)nGlobalNodes;
        S.topoDirty = true;                     // ghost rows get their reserved pattern id at the next finalize
        return SF3D_OK;
    }, (uint8_t)SF3D_SOLVER_ERROR);
}
void *sf3d_ext_stream(void) { return guarded([&]() -> void * { return dev_stream(); }, (void *)nullptr); }
uint8_t sf3d_ext_profile(int enable)
{ return guarded([&]() -> uint8_t { prof_enable(enable != 0); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR); }
uint8_t sf3d_ext_get_kernel_times(sf3d_kernel_times *out)
{
    if (!out) return SF3D_PARAMETER_ERROR;
    return guarded([&]() -> uint8_t { prof_get(out->ms, out->launches); return SF3D_OK; }, (uint8_t)SF3D_SOLVER_ERROR);
}

}  // extern "C"
