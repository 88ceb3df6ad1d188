// sf3d_rows.h -- per-node ("row") arithmetic of the water time step, written once as
// __host__ __device__ inline functions over SF3DView.  The CUDA kernels in sf3d_kernels.cu are
// thin grid-stride wrappers (index + block reduction) around these.
//
// Every function names the reference routine it replaces.  Operation order follows the
// reference expression by expression so that the only differences from the CPU solve are libm
// (CUDA pow/log/cbrt vs glibc) and reduction order; the library is compiled with -fmad=false.
#pragma once
#include <math.h>
#include <float.h>
#include "sf3d_view.h"

#define SF3D_EPSILON_METER   0.00001   // water.cpp:14
#define SF3D_EPSILON_RUNOFF  0.001     // commonConstants.h:267
#define SF3D_PI              3.1415926535898   // commonConstants.h:249

// Power function of the retention / conductivity curves (positive base).  The product build evaluates
// exp(y log x): about 2.5x fewer fp64 instructions than CUDA's pow() and within ~|y ln x| ulp of it
// (< 1e-14 relative for the arguments met here), far below the parity tolerances; the pow()-bound node
// kernels (Se, Mualem K) gain ~40 %.  -DSF3D_REFERENCE_ROUNDING keeps pow().
SF3D_HD double sf3d_pow(double x, double y)
{
#ifdef SF3D_DEVICE_MATH
    if (!(x > 0.)) return pow(x, y);            // zero / negative / NaN base: the library's special cases
    return exp(y * log(x));
#else
    return pow(x, y);
#endif
}

SF3D_HD double sf3d_max(double a, double b) { return (a < b) ? b : a; }   // std::max
SF3D_HD double sf3d_min(double a, double b) { return (b < a) ? b : a; }   // std::min

// ---- Math::computeMean (otherFunctions.cpp:7-37) ------------------------------------------
SF3D_HD double sf3d_mean(double v1, double v2, int type)
{
    if (type == 0) return (v1 + v2) * 0.5;                                   // arithmetic
    if (type == 1) { int sg = (v1 > 0) - (v1 < 0); return sg * sqrt(v1 * v2); }   // geometric
    return (v1 == v2) ? v1 : (v1 - v2) / log(v1 / v2);                       // logarithmic
}

// ---- Soil::computeNodeSe_fromPsi (soilPhysics.cpp:91-115) ---------------------------------
SF3D_HD double sf3d_se_from_psi(const SoilRec &s, int model, double psi)
{
    if (model == 0)   // VanGenuchten
        return sf3d_pow(1.0 + sf3d_pow(s.alpha * psi, s.n), -s.m);
    if (model == 1)   // ModifiedVanGenuchten
    {
        if (psi <= s.he) return 1.0;
        return sf3d_pow(1.0 + sf3d_pow(s.alpha * psi, s.n), -s.m) * s.invSc;
    }
    return SF3D_NODATA;
}

// ---- Soil::computeNodeSe (soilPhysics.cpp:69-85) ------------------------------------------
SF3D_HD double sf3d_node_se(const SoilRec &s, int model, double H, double z)
{
    if (H >= z) return 1.0;
    return sf3d_se_from_psi(s, model, fabs(H - z));
}

// ---- Soil::computeNodeTheta_fromSe / _fromSignedPsi (soilPhysics.cpp:38-63) ---------------
SF3D_HD double sf3d_theta_from_se(const SoilRec &s, double Se) { return (Se * (s.thetaS - s.thetaR)) + s.thetaR; }
SF3D_HD double sf3d_theta_from_signed_psi(const SoilRec &s, int model, double signedPsi)
{
    if (signedPsi >= 0.) return s.thetaS;
    return sf3d_theta_from_se(s, sf3d_se_from_psi(s, model, fabs(signedPsi)));
}

// ---- Soil::computeMualemSoilConductivity (soilPhysics.cpp:181-214) ------------------------
// sf3d_pow(Sc,1/m) and tDen depend on the soil only and are hoisted into SoilRec.
SF3D_HD double sf3d_mualem(const SoilRec &s, int model, double Se)
{
    if (Se >= 1.0) return s.Ksat;
    double temp;
    if (model == 0)
    {
        double SePow = sf3d_pow(Se, s.invM);
        temp = 1.0 - sf3d_pow(1.0 - SePow, s.m);
    }
    else if (model == 1)
    {
        double SeScPow = sf3d_pow(Se * s.Sc, s.invM);
        double tNum = 1.0 - sf3d_pow(1.0 - SeScPow, s.m);
        temp = tNum / s.tDen;
    }
    else
        return SF3D_NODATA;
#ifndef SF3D_REFERENCE_ROUNDING
    if (s.L == 0.5) return s.Ksat * sqrt(Se) * (temp * temp);      // Mualem's L = 0.5: exact square root
#endif
    return s.Ksat * sf3d_pow(Se, s.L) * (temp * temp);
}

// ---- Soil::computeNode_dTheta_dH (soilPhysics.cpp:224-279) --------------------------------
// SeCurr / SePrev are the stored saturation degrees of H and oldH: computeNodeSe_fromPsi of
// psiCurr / psiPrev returns exactly those values (same function, same arguments; psi = 0 gives
// 1), so the two pow pairs of the secant branch are not recomputed.
SF3D_HD double sf3d_dtheta_dh(const SoilRec &s, int model, double H, double oldH, double z,
                             double SeCurr, double SePrev)
{
    const double psiCurr = fabs(sf3d_min(0.0, H - z));
    const double psiPrev = fabs(sf3d_min(0.0, oldH - z));
    if (model == 0) { if (psiCurr == 0.0 && psiPrev == 0.0) return 0.0; }
    else if (model == 1) { if (psiCurr <= s.he && psiPrev <= s.he) return 0.0; }

    double dSe_dH;
    if (fabs(psiCurr - psiPrev) < 1e-12)
    {
        const double xx = s.alpha * psiCurr;
        const double onePlus = 1. + sf3d_pow(xx, s.n);
        const double term1 = sf3d_pow(onePlus, -(s.m + 1.));
        const double term2 = sf3d_pow(xx, s.n - 1.);
        dSe_dH = s.alpha * s.n * s.m * term1 * term2;
        if (model == 1) dSe_dH *= s.invSc;
    }
    else
        dSe_dH = fabs((SeCurr - SePrev) / (H - oldH));
    return dSe_dH * (s.thetaS - s.thetaR);
}

// ==========================================================================================
// begin of a try: CPUSolver::waterMainLoop body (cpusolver.cpp:155-169)
//   oldH = H ; x = H ; Se[soil] = computeNodeSe
// ==========================================================================================
SF3D_HD void sf3d_row_begin_try(const SF3DView &v, uint32_t i)
{
    const double H = v.H[i];
    v.oldH[i] = H;
    v.x0[i] = H;
    if (i < v.Ns)
        v.cap[i] = v.size[i];                      // surface capacity = cell area (cpusolver.cpp:151)
    else
    {
        const double se = sf3d_node_se(v.soil[v.tab[i]], v.wrcModel, H, v.z[i]);
        v.Se[i] = se;
        v.SeOld[i] = se;
    }
}

// restore after a refused try (cpusolver.cpp:182-186); Se is refreshed by the next begin_try
SF3D_HD void sf3d_row_restore_old(const SF3DView &v, uint32_t i) { v.H[i] = v.oldH[i]; }

// ==========================================================================================
// node phase of one approximation:
//   Water::computeCapacity (water.cpp:279-297) + Water::updateBoundaryWaterData (water.cpp:632-807)
// Heat hooks (vapour conductivity, HeatSurface evaporation) live in sf3d_rows_heat.h.
// ==========================================================================================
SF3D_HD double sf3d_heat_node_water(const SF3DView &v, uint32_t i, const SoilRec &s, double H, double z, double Se, double K,
                                   const double *dThetadH, double *dThetaVdH);
SF3D_HD double sf3d_heat_surface_boundary(const SF3DView &v, uint32_t i, double dt, double *upExtra);
SF3D_HD double sf3d_heat_surface_pull(const SF3DView &v, uint32_t i, double dt, int *active);

SF3D_HD double sf3d_culvert_flow(double waterLevel, double pond, double width, double height, double rough,
                                double slope, double bSize)
{
    // water.cpp:763-792 (pressure / mixed / open-channel regimes)
    double flow = 0.;
    if (waterLevel >= 1.5 * height)
    {
        double eqDiam = sqrt(4. * width * height / SF3D_PI);
        flow = (70. * pow(slope, 0.54)) * pow(eqDiam, 2.63) / 3.591;
    }
    else if (waterLevel >= height)
    {
        double wetted = width + 2. * height;
        double hydRadius = bSize / wetted;
        double manning = (bSize / rough) * sqrt(slope) * pow(hydRadius, 2. / 3.);
        double eqDiam = sqrt(4. * width * height / SF3D_PI);
        double pressure = (70. * pow(slope, 0.54)) * pow(eqDiam, 2.63) / 3.591;
        double weight = (waterLevel - height) / (0.5 * height);
        flow = weight * pressure + (1. - weight) * manning;
    }
    else if (waterLevel > pond)
    {
        double bArea = width * waterLevel;
        double wetted = width + 2. * waterLevel;
        double hydRadius = bArea / wetted;
        flow = (bArea / rough) * sqrt(slope) * pow(hydRadius, 2. / 3.);
    }
    return flow;
}

// pond of a node as the reference stores it: per node, NODATA on soil nodes (soilFluxes3D.cpp:616); the device
// array has surface entries only, so a Runoff type on a soil node must not index it
SF3D_HD double sf3d_pond(const SF3DView &v, uint32_t i) { return (i < v.Ns) ? v.pond[i] : SF3D_NODATA; }

// HEAT is a compile-time switch so that the water-only kernels carry none of the heat closures
template <bool HEAT>
SF3D_HD void sf3d_row_node_phase(const SF3DView &v, uint32_t i, double dt, int withCapacity)
{
    const uint32_t m = v.meta[i];
    const bool surface = META_SURFACE(m);
    const double H = v.H[i], oldH = v.oldH[i], z = v.z[i];

    double K = 0.;
    if (!surface)
    {
        const SoilRec &s = v.soil[v.tab[i]];
        const double Se = v.Se[i];
        // computeNodeK (soilPhysics.cpp:164-172)
        K = sf3d_mualem(s, v.wrcModel, Se);
        double dThetadH = 0., dThetaVdH = 0.;
        if (withCapacity) dThetadH = sf3d_dtheta_dh(s, v.wrcModel, H, oldH, z, Se, v.SeOld[i]);
        if (HEAT) K = sf3d_heat_node_water(v, i, s, H, z, Se, K, withCapacity ? &dThetadH : nullptr, &dThetaVdH);
        v.K[i] = K;
        if (withCapacity)
        {
            double c = v.size[i] * dThetadH;
            if (HEAT && v.computeHeatVapor) c += v.size[i] * dThetaVdH;
            v.cap[i] = c;
        }
    }

    // ---- updateBoundaryWaterData (water.cpp:639-806) ----
    double flow = v.sink[i];
    if (surface && flow < 0)
    {
        const double avgH = 0.5 * (H + oldH);
        const double hs = sf3d_max(0., avgH - z);
        const double maxSurfaceFlux = -hs * v.size[i] / dt;
        flow = sf3d_max(flow, maxSurfaceFlux);
    }
    // HeatSurface surface-water evaporation, pulled by the surface node through its Down link.
    // The reference writes it from the soil node's iteration (water.cpp:722-736, order dependent
    // under OpenMP, SURVEY Q9); the sequential order is reproduced: applied after the node's own terms.
    int evapActive = 0;
    double surfEvap = 0.;
    if (HEAT && surface && v.computeHeatVapor) surfEvap = sf3d_heat_surface_pull(v, i, dt, &evapActive);

    const uint32_t bt = META_BT(m);
    if (bt == BT_NONE)
    {
        if (evapActive) flow += surfEvap;                             // water.cpp:735
        v.wFlow[i] = flow;
        return;
    }

    double rate = 0.;
    switch (bt)
    {
        case BT_RUNOFF:
        {
            const double avgH = 0.5 * (H + oldH);
            const double hs = sf3d_max(0., avgH - (z + sf3d_pond(v, i)));
            if (hs < SF3D_EPSILON_RUNOFF) break;
            const double maxFlow = (hs * v.size[i]) / dt;
            const double vel = pow(hs, 2. / 3.) * sqrt(v.bSlope[i]) / v.rough[v.tab[i]];
            const double valFlow = hs * vel * v.bSize[i];
            rate = -sf3d_min(valFlow, maxFlow);
            break;
        }
        case BT_FREE_DRAINAGE:
            rate = -K * v.larea[i];                                   // slot 0 (Up) interface area
            break;
        case BT_FREE_LATERAL:
            rate = -K * v.bSize[i] * v.bSlope[i] * v.lvRatio;
            break;
        case BT_PRESCRIBED:
        {
            const SoilRec &s = v.soil[v.tab[i]];
            const double L = 1.;
            const double boundaryZ = z - L;
            const double boundaryPsi = v.bPresc[i] - boundaryZ;
            const double boundaryK = (boundaryPsi >= 0) ? s.Ksat
                : sf3d_mualem(s, v.wrcModel, sf3d_se_from_psi(s, v.wrcModel, fabs(boundaryPsi)));
            const double meanK = sf3d_mean(boundaryK, K, v.meanType);
            const double dH = v.bPresc[i] - H;
            rate = meanK * v.bSize[i] * (dH / L);
            break;
        }
        case BT_HEAT_SURFACE:
            if (HEAT && v.computeHeatVapor) rate = sf3d_heat_surface_boundary(v, i, dt, nullptr);
            break;
        case BT_CULVERT:
        {
            // Reference water.cpp:749-795 is unreachable (culvertPtr never allocated) and uses
            // 0.5*(H - oldH) - z; the v1 code (old/old_boundary.cpp:377) used the mean head.  The
            // physical (v1) form is built here; see DESIGN.md "deviations".
            // a Culvert type set through setNode / setNodeBoundary without setCulvert has no record (the
            // reference would dereference a null pointer there): no flow
            const uint32_t rec = (v.culverts && v.culvertOf && i < v.Ns) ? v.culvertOf[i] : 0u;
            if (rec)
            {
                const CulvertRec c = v.culverts[rec - 1u];
                const double waterLevel = 0.5 * (H + oldH) - z;
                rate = -sf3d_culvert_flow(waterLevel, v.pond[i], c.width, c.height, c.roughness, v.bSlope[i], v.bSize[i]);
            }
            break;
        }
        default:        // Urban, Road, SoluteFlux: water.cpp:796-799
            rate = 0.;
            break;
    }
    if (fabs(rate) < DBL_EPSILON) rate = 0.;
    else flow += rate;
    if (evapActive) rate = surfEvap;                                  // water.cpp:732-733: overwrites the rate only
    v.bRate[i] = rate;
    v.wFlow[i] = flow;
}

// ==========================================================================================
// link conductances: Water::computeLinkFluxes dispatch (water.cpp:300-343)
// ==========================================================================================

// Water::redistribution (water.cpp:542-562).
// Reference: cellDistance = 3-D distance (lateral) or |dz| (vertical); lateral K scaled by the
// horizontal/vertical ratio; (mean(Ki,Kj) * area) / distance.
// Product build: the static factor geom = area / distance (x ratio for lateral links; every mean is
// homogeneous of degree 1) is precomputed per link by kern_link_geometry, which removes one fp64
// division, two multiplications and one 8-byte load per link; the result differs from the
// reference expression by rounding only (<= 2 ulp).  -DSF3D_REFERENCE_ROUNDING keeps the
// reference's exact expression (geom then holds the distance).
SF3D_HD double sf3d_redistribution(const SF3DView &v, double ki, double kj, int slot, double area, double geom)
{
#ifdef SF3D_REFERENCE_ROUNDING
    if (geom == 0.) return 0.;
    if (slot >= 2) { ki *= v.lvRatio; kj *= v.lvRatio; }
    return (sf3d_mean(ki, kj, v.meanType) * area) / geom;
#else
    (void)slot; (void)area;
    return sf3d_mean(ki, kj, v.meanType) * geom;
#endif
}

// Water::infiltration (water.cpp:490-539); dist = z[surface] - z[soil]
SF3D_HD double sf3d_infiltration(const SF3DView &v, uint32_t surf, uint32_t soil, double dt, double area, double dist)
{
    const SoilRec &s = v.soil[v.tab[soil]];
    double boundaryFactor = 1.;
    const uint32_t bt = META_BT(v.meta[soil]);
    if (bt == BT_URBAN) boundaryFactor = 0.33;
    else if (bt == BT_ROAD) return 0.;

    if (v.H[soil] > v.z[surf])
        return (s.Ksat * boundaryFactor * area) / dist;

    const double surfH = 0.5 * (v.H[surf] + v.oldH[surf]);
    const double soilH = 0.5 * (v.H[soil] + v.oldH[soil]);
    double surfaceWater = sf3d_max(surfH - v.z[surf], 0.);
    const double surfaceBoundaryFlow = v.wFlow[surf];
    if (surfaceBoundaryFlow < 0.)
    {
        const double boundary_m = (surfaceBoundaryFlow * dt) / v.size[surf];
        surfaceWater = sf3d_max(0., surfaceWater + boundary_m);
    }
    const double maxInfRate = surfaceWater / dt;
    if (maxInfRate < 2.78e-11) return 0.;

    const double dH = sf3d_max(surfH - soilH, 1e-12);
    const double maxK = maxInfRate * (dist / dH);
    const double meanK = sf3d_mean(s.Ksat, v.K[soil], v.meanType);
    return (sf3d_min(boundaryFactor * meanK, maxK) * area) / dist;
}

// Water::runoffConductance (water.cpp:413-487); dist = 2-D distance; updates the row's Courant
SF3D_HD double sf3d_runoff(const SF3DView &v, uint32_t i, uint32_t j, int approx, double dt, double flowSide,
                          double dxy, double *courant)
{
    double Hi = 0.5 * (v.H[i] + v.oldH[i]);
    double Hj = 0.5 * (v.H[j] + v.oldH[j]);
    if (approx == 0)
    {
        const double wi = v.wFlow[i], wj = v.wFlow[j];
        if (wi > 0) Hi += 0.5 * wi * dt / v.size[i];
        if (wj > 0) Hj += 0.5 * wj * dt / v.size[j];
    }
    const double zi = v.z[i] + v.pond[i];
    const double zj = v.z[j] + v.pond[j];
    const double Hmax = sf3d_max(Hi, Hj);
    const double zmax = sf3d_max(zi, zj);
    const double Hs = Hmax - zmax;
    if (Hs <= SF3D_EPSILON_METER) return 0.0;
    if (dxy <= 0.0) return 0.0;
    const double roughness = 0.5 * (v.rough[v.tab[i]] + v.rough[v.tab[j]]);
    if (roughness <= 0.0) return 0.0;

    const double A = flowSide * Hs;
    const double Hs23 = cbrt(Hs * Hs);
    const double Kij = A * Hs23 / (roughness * dxy);

    const double dH = fabs(Hi - Hj);
    const double slope = (dH > SF3D_EPSILON_METER) ? dH / dxy : 0.0;
    const double vel = Hs23 * sqrt(slope) / roughness;
    *courant = sf3d_max(*courant, vel * dt / dxy);
    return Kij;
}

SF3D_HD double sf3d_heat_thermal_invariant(const SF3DView &v, uint32_t i, int slot, const SF3DPair tli, const SF3DPair tvi, double tmi,
                                          const SF3DPair tlj, const SF3DPair tvj, double tmj);   // water.cpp:329-340
SF3D_HD SF3DPair h_pair_load(const double *arr, uint32_t i);

// ==========================================================================================
// assembly of one row: CPUSolver::computeLinearSystemElement + computeDiagonalElement +
// preconditioningMatrix (cpusolver.cpp:348-389, 335-345, 284-305).  Returns the row's Courant.
// Columns are visited in the reference's order (Up, Lateral 0..7, Down).  v.mcol[c] is the linked
// node of column c, or the row itself when the link does not exist (then geom = 0).
// ==========================================================================================
SF3D_HD void sf3d_row_store(const SF3DView &v, uint32_t i, double dt, const double *k, int kstride, double sum, double invariant)
{
    const size_t N = v.N;
    const double capOverDt = v.cap[i] / dt;
    const double diag = capOverDt + sum;              // cpusolver.cpp:344
    const double invDiag = 1.0 / diag;                // cpusolver.cpp:291
    #pragma unroll
    for (int c = 0; c < SF3D_NLINK; ++c)
        v.mval[(size_t)c * N + i] = (-k[c * kstride]) * invDiag;     // cpusolver.cpp:380-383, 294-297
    const double rhs = (capOverDt * v.oldH[i]) + v.wFlow[i] + invariant;   // :387-388 (invariant = 0 without heat)
    v.b[i] = rhs * invDiag;                           // cpusolver.cpp:300
}

// linked nodes of the ten matrix columns of row i.  With pattern compression: the most frequent
// pattern (interior nodes, > 95 % of a DEM catchment) comes from kernel parameters (no memory access at
// all), other rows read their ten offsets from the small pattern table; without: the explicit array.
SF3D_HD void sf3d_row_cols(const SF3DView &v, uint32_t i, uint32_t *j)
{
    if (v.pattern)
    {
        const uint32_t p = v.pid[i] & SF3D_PID_MASK;
        if (p == v.hotPid)
        {
            #pragma unroll
            for (int c = 0; c < SF3D_NLINK; ++c) j[c] = (uint32_t)((int64_t)i + v.hotOff[c]);
        }
        else
        {
            const int32_t *off = v.pattern + (size_t)p * SF3D_NLINK;
            #pragma unroll
            for (int c = 0; c < SF3D_NLINK; ++c) j[c] = (uint32_t)((int64_t)i + off[c]);
        }
    }
    else
    {
        #pragma unroll
        for (int c = 0; c < SF3D_NLINK; ++c) j[c] = v.mcol[(size_t)c * v.N + i];
    }
}

// assembly variant: one pointer to the row's ten offsets (fewer live registers than the branchy form,
// and the assembly kernel is bound by fp64 issue, not by these L1-resident loads)
SF3D_HD const int32_t *sf3d_row_pattern(const SF3DView &v, uint32_t i)
{
    return v.pattern ? v.pattern + (size_t)(v.pid[i] & SF3D_PID_MASK) * SF3D_NLINK : nullptr;
}
SF3D_HD uint32_t sf3d_col_index(const SF3DView &v, const int32_t *__restrict__ off, uint32_t i, int c)
{
    return off ? (uint32_t)((int64_t)i + off[c]) : v.mcol[(size_t)c * v.N + i];
}

// soil row: every link is a redistribution except an Up link to a surface node (infiltration).
// The ten neighbour conductivities are gathered first (independent loads), then the means.
template <bool HEAT>
SF3D_HD double sf3d_row_assemble_soil(const SF3DView &v, uint32_t i, double dt, double *k, int kstride)
{
    // k: per-thread scratch for the ten conductances (shared memory on the device: keeps them out of the
    // register file so that more warps are resident while the neighbour gathers are in flight)
    const size_t N = v.N;
    const double ki = v.K[i];
    const int32_t *off = sf3d_row_pattern(v, i);
    double sum = 0.;
    // links are handled in two groups of five: all gathers of a group are issued before its arithmetic
    // (independent loads in flight)
    #pragma unroll
    for (int half = 0; half < 2; ++half)
    {
        uint32_t j[5];
        double g[5], kj[5];
        #pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            const int c = half * 5 + q;
            j[q] = sf3d_col_index(v, off, i, c);
            g[q] = SF3D_LDS(v.lgeom + (size_t)c * N + i);
        }
        #pragma unroll
        for (int q = 0; q < 5; ++q) kj[q] = v.K[j[q]];
        #pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            const int c = half * 5 + q;
            const int slot = sf3d_slot_of_col(c);
            double kc;
            if (c == 0 && j[0] < v.Ns)                    // first soil layer: link to the surface node above
                kc = sf3d_infiltration(v, j[0], i, dt, v.larea[i], g[0]);
            else
            {
#ifdef SF3D_REFERENCE_ROUNDING
                const double area = v.larea[(size_t)slot * N + i];
#else
                const double area = 0.;
#endif
                kc = sf3d_redistribution(v, ki, kj[q], slot, area, g[q]);
            }
            k[c * kstride] = kc;
            sum += kc;                                    // zero entries are not stored in the reference; +0 is exact
        }
    }
    // with the heat coupling: the row's thermal liquid / vapour fluxes (water.cpp:329-340), summed in the same link
    // order by sf3d_row_thermal_invariant (its own pass: it needs few registers, this one many)
    const double invariant = HEAT ? v.hInv[i] : 0.;
    sf3d_row_store(v, i, dt, k, kstride, sum, invariant);
    return 0.;
}

// surface row: runoff links to surface neighbours, infiltration link to the soil node below
SF3D_HD double sf3d_row_assemble_surface(const SF3DView &v, uint32_t i, double dt, int approx, double *k, int kstride)
{
    const size_t N = v.N;
    const uint32_t m = v.meta[i];
    double sum = 0., courant = 0.;
    #pragma unroll
    for (int c = 0; c < SF3D_NLINK; ++c)
    {
        const int slot = sf3d_slot_of_col(c);
        double kc = 0.;
        if (META_HAS_SLOT(m, slot))
        {
            const uint32_t j = v.mcol[(size_t)c * N + i];
            const double area = v.larea[(size_t)slot * N + i];
            const double dist = v.lgeom[(size_t)c * N + i];
            if (j < v.Ns) kc = sf3d_runoff(v, i, j, approx, dt, area, dist, &courant);
            else          kc = sf3d_infiltration(v, i, j, dt, area, dist);
        }
        k[c * kstride] = kc;
        sum += kc;
    }
    sf3d_row_store(v, i, dt, k, kstride, sum, 0.);
    return courant;
}

template <bool HEAT>
SF3D_HD double sf3d_row_assemble(const SF3DView &v, uint32_t i, double dt, int approx, double *k, int kstride)
{
    return (i < v.Ns) ? sf3d_row_assemble_surface(v, i, dt, approx, k, kstride) : sf3d_row_assemble_soil<HEAT>(v, i, dt, k, kstride);
}

// ==========================================================================================
// Water::JacobiWaterCPU, one row (water.cpp:570-596).  Returns the row's contribution to the norm.
// COHERENT: the row of the persistent small-graph solve (all sweeps of a solve in ONE kernel, grid-wide barrier
// between sweeps): the solution vectors are written by other thread blocks earlier in the same launch, so they are
// read through L2 (ld.global.cg) and never through the non-coherent read-only path.  Same operations in the same order.
// ==========================================================================================
#if defined(__CUDA_ARCH__)
#define SF3D_LDCG(p) __ldcg(p)
#else
#define SF3D_LDCG(p) (*(p))
#endif
template <bool COHERENT = false>
SF3D_HD double sf3d_row_jacobi(const SF3DView &v, uint32_t i, const double *__restrict__ xin, double *__restrict__ xout,
                               double *xnewOut = nullptr)
{
    const size_t N = v.N;
    uint32_t j[SF3D_NLINK];
    sf3d_row_cols(v, i, j);
    double xnew = SF3D_LDS(v.b + i);
    #pragma unroll
    for (int c = 0; c < SF3D_NLINK; ++c)
    {
        const double A = SF3D_LDS(v.mval + (size_t)c * N + i);
        xnew -= A * (COHERENT ? SF3D_LDCG(xin + j[c]) : xin[j[c]]);
    }
    const double z = SF3D_LDS(v.z + i);
    if (i < v.Ns) xnew = sf3d_max(xnew, z);
    const double xold = COHERENT ? SF3D_LDCG(xin + i) : xin[i];
    double norm = fabs(xnew - xold);
    const double psi = fabs(xnew - z);
    if (psi > 1.) norm *= (1. / psi);
    xout[i] = xnew;
    if (xnewOut) *xnewOut = xnew;
    return norm;
}

// ==========================================================================================
// after the solve (cpusolver.cpp:451-457) fused with Water::computeCurrentMassBalance's two
// reductions (water.cpp:71-90, 130-140): H = x ; Se[soil] ; storage_i ; sink_i
// ==========================================================================================
SF3D_HD void sf3d_row_post(const SF3DView &v, uint32_t i, const double *__restrict__ x, double dt,
                          int mode, double *storage, double *sinkFlow)
{
    // mode 0: after a solve (H = x, Se recomputed); mode 1: H kept, Se recomputed;
    // mode 2: stored Se used as is (Water::computeTotalWaterContent, water.cpp:71-90)
    double H;
    if (mode == 0) { H = x[i]; v.H[i] = H; } else H = v.H[i];
    const double z = v.z[i];
    double theta;
    if (i < v.Ns)
        theta = sf3d_max(H - z, 0.0);
    else
    {
        const SoilRec &s = v.soil[v.tab[i]];
        double se;
        if (mode == 2) se = v.Se[i];
        else { se = sf3d_node_se(s, v.wrcModel, H, z); v.Se[i] = se; }
        theta = sf3d_theta_from_se(s, se);
    }
    *storage = theta * v.size[i];
    const double wf = v.wFlow[i];
    *sinkFlow = (wf != 0) ? wf * dt : 0.;
}

// ==========================================================================================
// Water::acceptStep per node (water.cpp:240-250) with updateLinkFlux (water.cpp:269-277).
// The reference multiplies the NORMALISED off-diagonal by the diagonal slot, which
// preconditioningMatrix has already overwritten with 1.0 (cpusolver.cpp:303, cpusolver.h:51):
// the accumulated link flow is A'_ij (H_i - H_j) dt with A'_ij = -k_ij / D_i.  Reproduced as is
// (SURVEY Appendix B, Q1).  Links whose conductance was 0 contribute 0 (Q2).
// ==========================================================================================
SF3D_HD void sf3d_row_accept(const SF3DView &v, uint32_t i, double dt)
{
    const size_t N = v.N;
    const uint32_t m = v.meta[i];
    const double Hi = v.H[i];
    // linked nodes from the row's link pattern (an existing link's matrix column is its link index; absent links have
    // a zero entry and are skipped), so the explicit 4-byte link index array is not read
    uint32_t j[SF3D_NLINK];
    sf3d_row_cols(v, i, j);
    #pragma unroll
    for (int c = 0; c < SF3D_NLINK; ++c)
    {
        const int slot = sf3d_slot_of_col(c);
        if (!META_HAS_SLOT(m, slot)) continue;
        const double A = v.mval[(size_t)c * N + i];
        if (A == 0.) continue;
        v.lflow[(size_t)slot * N + i] += A * (Hi - v.H[j[c]]) * dt;
    }
    if (META_BT(m) != BT_NONE) v.bSum[i] += v.bRate[i] * dt;
}

// what the next try's first pass would do (sf3d_row_begin_try), done while the accepted state is at hand: after an
// accepted step the stored Se IS computeNodeSe(H) (written by the post pass or by restore-best from the same H), so
// the pass reduces to copies.  The engine skips kern_begin_try while nothing has touched the state in between.
SF3D_HD void sf3d_row_prepare_try(const SF3DView &v, uint32_t i)
{
    const double H = v.H[i];
    v.oldH[i] = H;
    v.x0[i] = H;
    if (i < v.Ns) v.cap[i] = v.size[i];
    else v.SeOld[i] = v.Se[i];
}

// Water::restoreBestStep per node (water.cpp:255-263): H = best ; Se ; K
SF3D_HD void sf3d_row_restore_best(const SF3DView &v, uint32_t i)
{
    const double H = v.bestH[i];
    v.H[i] = H;
    if (i >= v.Ns)
    {
        const SoilRec &s = v.soil[v.tab[i]];
        const double se = sf3d_node_se(s, v.wrcModel, H, v.z[i]);
        v.Se[i] = se;
        // K is recomputed by the boundary pass that follows (node phase without capacity)
    }
}

// ==========================================================================================
// static link geometry (Soil::nodeDistance2D/3D, soilPhysics.cpp:325-335; water.cpp:500,550,557)
// ==========================================================================================
SF3D_HD double sf3d_link_distance(const SF3DView &v, uint32_t i, uint32_t j, int slot)
{
    const bool iS = i < v.Ns, jS = j < v.Ns;
    const double dx = v.x[i] - v.x[j], dy = v.y[i] - v.y[j], dz = v.z[i] - v.z[j];
    if (!iS && !jS)
    {
        if (slot >= 2) { double n = 0; n += dx * dx; n += dy * dy; n += dz * dz; return sqrt(n); }
        return fabs(dz);
    }
    if (iS && jS) { double n = 0; n += dx * dx; n += dy * dy; return sqrt(n); }
    return iS ? dz : -dz;           // z[surface] - z[soil]
}

// what v.lgeom holds for link (i -> j): the distance, except soil-soil links of the product build,
// which hold area / distance (x horizontal/vertical ratio for lateral links); see sf3d_redistribution
SF3D_HD double sf3d_link_geom(const SF3DView &v, uint32_t i, uint32_t j, int slot, double area)
{
    const double d = sf3d_link_distance(v, i, j, slot);
#ifndef SF3D_REFERENCE_ROUNDING
    if (i >= v.Ns && j >= v.Ns)
    {
        const double g = area / d;
        return (slot >= 2) ? g * v.lvRatio : g;
    }
#else
    (void)area;
#endif
    return d;
}
