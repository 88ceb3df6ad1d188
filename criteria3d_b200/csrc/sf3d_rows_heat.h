// sf3d_rows_heat.h -- coupled heat transport: the closures of agrolib/soilFluxes3D/heat.cpp as
// __host__ __device__ functions, the heat-coupling hooks of the water rows (vapour conductivity,
// thermal liquid/vapour fluxes, HeatSurface evaporation) and the rows of the heat update itself.
// Every function cites the reference lines it replaces; operation order follows the reference.
#pragma once
#include "sf3d_rows.h"

// commonConstants.h
#define HC_GRAVITY 9.80665
#define HC_WATER_DENSITY 1000.
#define HC_MH2O 0.018
#define HC_ZEROCELSIUS 273.15
#define HC_R_GAS 8.31447215
#define HC_R_DRY_AIR 287.058
#define HC_LAPSE_RATE_MOIST_AIR 0.0065
#define HC_P0 101325.
#define HC_TP0 293.16
#define HC_GAMMA0 71.89
#define HC_MINERAL_HK 2.5
#define HC_VON_KARMAN 0.41
#define HC_QUARTZ_DENSITY 2.648
#define HC_HEAT_CAPACITY_WATER 4182000.
#define HC_HEAT_CAPACITY_AIR 1290.
#define HC_HEAT_CAPACITY_MINERAL 231000.
#define HC_HEAT_CAPACITY_WATER_VAPOR 1996.
#define HC_HEAT_CAPACITY_AIR_MOLAR 29.31
#define HC_VAPOR_DIFFUSIVITY0 0.0000212
#define HC_THETAMIN 0.15

#ifndef SF3D_HEAT_LINK_UNROLL
#define SF3D_HEAT_LINK_UNROLL 1      // link loops of the heat rows
#endif
constexpr int kHeatLinkUnroll = SF3D_HEAT_LINK_UNROLL;
#ifndef SF3D_THERMAL_UNROLL
#define SF3D_THERMAL_UNROLL 5        // link loops of the thermal invariant fluxes: two groups of five links (A/B on B200, two-pass form:
                                     // unroll 1 / 2 / 5 / 10 -> 2.01 / 1.80 / 1.59 / 1.71 ms per approximation for this pass + the assembly)
#endif
constexpr int kThermalUnroll = SF3D_THERMAL_UNROLL;
#ifndef SF3D_HEAT_ACCEPT_UNROLL
#define SF3D_HEAT_ACCEPT_UNROLL 1    // link loop of saveNodeHeatFluxes
#endif
constexpr int kHeatAcceptUnroll = SF3D_HEAT_ACCEPT_UNROLL;

// pow() with the small integer exponents heat.cpp passes: the product multiplies, the reference-rounding
// build calls the library like the reference does
#ifdef SF3D_DEVICE_MATH
SF3D_HD double h_pow1(double x) { return x; }
SF3D_HD double h_pow2(double x) { return x * x; }
SF3D_HD double h_pow3(double x) { return x * x * x; }
SF3D_HD double h_pow4(double x) { const double x2 = x * x; return x2 * x2; }
#else
SF3D_HD double h_pow1(double x) { return pow(x, 1.); }
SF3D_HD double h_pow2(double x) { return pow(x, 2.); }
SF3D_HD double h_pow3(double x) { return pow(x, 3); }
SF3D_HD double h_pow4(double x) { return pow(x, 4); }
#endif

// ---- small closures (heat.cpp:1043-1250) ----------------------------------------------------
SF3D_HD double h_latent_vaporization(double Tc) { return (2501000. - 2369.2 * Tc); }                    // :1085
SF3D_HD double h_sat_vapor_pressure(double Tc) { return 611 * exp(17.502 * Tc / (Tc + 240.97)); }       // :1164
SF3D_HD double h_vapor_conc_from_pressure(double p, double T) { return (p * HC_MH2O / (HC_R_GAS * T)); }   // :1219
SF3D_HD double h_vapor_pressure_from_conc(double c, double T) { return (c * HC_R_GAS * T / HC_MH2O); }     // :1208
SF3D_HD double h_soil_relative_humidity(double h, double T) { return exp(HC_MH2O * h * HC_GRAVITY / (HC_R_GAS * T)); }   // :1144
SF3D_HD double h_vapor_from_psi_temp(double h, double T)                                                 // :1071
{
    const double svp = h_sat_vapor_pressure(T - HC_ZEROCELSIUS);
    const double svc = h_vapor_conc_from_pressure(svp, T);
    const double rh = h_soil_relative_humidity(h, T);
    return svc * rh;
}
SF3D_HD double h_pressure_from_altitude(double height)                                                    // :1117
{ return HC_P0 * sf3d_pow(1 + height * HC_LAPSE_RATE_MOIST_AIR / HC_TP0, -HC_GRAVITY / (HC_LAPSE_RATE_MOIST_AIR * HC_R_DRY_AIR)); }
SF3D_HD double h_air_molar_density(double p, double T) { return 44.65 * (p / HC_P0) * (HC_ZEROCELSIUS / T); }   // :1186
SF3D_HD double h_air_vol_specific_heat(double p, double T) { return HC_HEAT_CAPACITY_AIR_MOLAR * h_air_molar_density(p, T); }   // :1197
SF3D_HD double h_svp_slope(double Tc, double svp) { return (4098. * svp / ((237.3 + Tc) * (237.3 + Tc))); }   // :1175
SF3D_HD double h_vapor_binary_diffusivity(double T) { return HC_VAPOR_DIFFUSIVITY0 * h_pow2(T / HC_ZEROCELSIUS); }   // :1230
SF3D_HD double h_soil_vapor_diffusivity(double thetaS, double theta, double T)                            // :1127
{
    const double beta = 0.66, m = 1.;
    (void)m;
    return h_vapor_binary_diffusivity(T) * beta * h_pow1(thetaS - theta);
}
SF3D_HD double h_soil_surface_resistance(double thetaTop) { return 10 * exp(0.3563 * (HC_THETAMIN - thetaTop) * 100); }   // :1154
SF3D_HD double h_water_return_flow_factor(double theta, double T, double clay)                            // :1097
{
    const double wc0 = 0.078 + 0.33 * clay;
    if (theta < 0.01 * wc0) return 0.;
    const double q0 = 2.52 + 7.25 * clay;
    const double q = q0 * h_pow2(T / 303.);
    return 1. / (1. + sf3d_pow(theta / wc0, -q));
}
SF3D_HD double h_thermal_liquid_conductivity(double Tc, double h, double ILK)                             // :1242
{
    const double Gwt = 4.;
    const double dGammadT = -0.1425 - 0.000576 * Tc;
    return sf3d_max(0., ILK * h * Gwt * dGammadT / HC_GAMMA0);
}
SF3D_HD double h_particle_density(double om)                                                              // :1057
{
    if (om == SF3D_NODATA) om = 0.02;
    return 1. / ((1. - om) / HC_QUARTZ_DENSITY + om / 1.43);
}
SF3D_HD double h_bulk_density(const SoilRec &s) { return (1. - s.thetaS) * h_particle_density(s.organicMatter); }   // :1043

// ---- node closures ------------------------------------------------------------------------------
SF3D_HD const SoilRec &h_soil(const SF3DView &v, uint32_t i) { return v.soil[v.tab[i]]; }
SF3D_HD double h_theta(const SF3DView &v, uint32_t i, double signedPsi)            // computeNodeTheta_fromSignedPsi
{ return (i < v.Ns) ? 1. : sf3d_theta_from_signed_psi(h_soil(v, i), v.wrcModel, signedPsi); }
SF3D_HD double h_mean_T(const SF3DView &v, uint32_t i) { return (v.T[i] + v.oldT[i]) * 0.5; }   // getNodeMeanTemperature, soilPhysics.cpp:305-311

// The vapour closures of one node share their sub-expressions (saturation vapour pressure and
// concentration, soil relative humidity, vapour diffusivity): evaluated once per (node, T, h) here, the
// closures below combine them with the reference's own operations in the reference's order.
struct HeatNodeCtx { double T, theta, svp, svc, rh, vConc, vDiff; };
SF3D_HD HeatNodeCtx h_node_ctx(const SoilRec &s, double T, double h, double theta)
{
    HeatNodeCtx c;
    c.T = T; c.theta = theta;
    c.svp = h_sat_vapor_pressure(T - HC_ZEROCELSIUS);
    c.svc = h_vapor_conc_from_pressure(c.svp, T);
    c.rh = h_soil_relative_humidity(h, T);
    c.vConc = c.svc * c.rh;                                          // VaporFromPsiTemp, heat.cpp:1071
    c.vDiff = h_soil_vapor_diffusivity(s.thetaS, theta, T);
    return c;
}
// computeNodeThermalVaporConductivity (heat.cpp:780-819); aPressure = pressureFromAltitude(z)
SF3D_HD double h_tvk(const SoilRec &s, const HeatNodeCtx &c, double aPressure)
{
    const double Tc = c.T - HC_ZEROCELSIUS;
    const double svpSlope = h_svp_slope(Tc, c.svp / 1000);
    const double svcSlope = svpSlope * HC_MH2O * h_air_molar_density(aPressure, c.T) / aPressure;
    const double vPressure = h_vapor_pressure_from_conc(c.vConc, c.T);
    const double rH = vPressure / c.svp;
    const double satDegree = c.theta / s.thetaS;
    const double eta = 9.5 + 3. * satDegree - 8.5 * exp(-h_pow4(s.etaClay * satDegree));
    return eta * c.vDiff * svcSlope * rH;
}
// computeNodeIsothermalVaporConductivity (heat.cpp:827-841)
SF3D_HD double h_ivk(const HeatNodeCtx &c) { return (c.vDiff * c.vConc * HC_MH2O) / (HC_R_GAS * c.T); }
// computeNodeHeatAirConductivity (heat.cpp:752-772); computeWater is always true on this path
SF3D_HD double h_air_conductivity(double T, double tvk)
{
    const double Tc = T - HC_ZEROCELSIUS;
    double aK = 0.024 + 0.0000773 * Tc - 0.000000026 * Tc * Tc;
    const double lambda = h_latent_vaporization(Tc);
    aK += lambda * tvk;
    return aK;
}
// computeNodeHeatSoilConductivity (heat.cpp:702-744); tvk = thermal vapour conductivity at (T, h)
SF3D_HD double h_soil_heat_conductivity(const SoilRec &s, const HeatNodeCtx &c, double tvk)
{
    const double T = c.T;
    const double Tc = T - HC_ZEROCELSIUS;
    const double wVol = c.theta;
    const double sVol = 1. - s.thetaS;
    const double aVol = s.thetaS - wVol;
    const double wRet = h_water_return_flow_factor(wVol, T, s.clay);
    const double wK = 0.554 + 0.0024 * Tc - 0.00000987 * Tc * Tc;
    const double aK = h_air_conductivity(T, tvk);
    const double fK = aK + wRet * (wK - aK);
    const double ga = 0.088;
    const double gc = 1. - 2. * ga;
    const double aW = (2. / (1. + (aK / fK - 1.) * ga) + 1. / (1. + (aK / fK - 1.) * gc)) / 3.;
    const double wW = (2. / (1. + (wK / fK - 1.) * ga) + 1. / (1. + (wK / fK - 1.) * gc)) / 3.;
    const double sW = (2. / (1. + (HC_MINERAL_HK / fK - 1.) * ga) + 1. / (1. + (HC_MINERAL_HK / fK - 1.) * gc)) / 3.;
    return (wVol * wW * wK + aVol * aW * aK + sVol * sW * HC_MINERAL_HK) / (wW * wVol + aW * aVol + sW * sVol);
}
// the same closures from (node, T, h), as the reference calls them.  The per-node pressure table lives on
// the device; the host getters (views over host mirrors, hPress == null) evaluate the closure
SF3D_HD double h_node_pressure(const SF3DView &v, uint32_t i) { return v.hPress ? v.hPress[i] : h_pressure_from_altitude(v.z[i]); }
SF3D_HD double h_thermal_vapor_conductivity(const SF3DView &v, uint32_t i, double T, double h)
{
    const SoilRec &s = h_soil(v, i);
    return h_tvk(s, h_node_ctx(s, T, h, h_theta(v, i, h)), h_node_pressure(v, i));
}
SF3D_HD double h_soil_heat_conductivity(const SF3DView &v, uint32_t i, double T, double h)
{
    const SoilRec &s = h_soil(v, i);
    const HeatNodeCtx c = h_node_ctx(s, T, h, h_theta(v, i, h));
    return h_soil_heat_conductivity(s, c, h_tvk(s, c, h_node_pressure(v, i)));
}
// computeNodeVaporThetaV (heat.cpp:868-875)
SF3D_HD double h_vapor_theta_v(const SF3DView &v, uint32_t i, double h, double T)
{
    const SoilRec &s = h_soil(v, i);
    const double theta = h_theta(v, i, h);
    return h_vapor_from_psi_temp(h, T) / HC_WATER_DENSITY * (s.thetaS - theta);
}
// computeNodeHeatCapacity (heat.cpp:849-860)
SF3D_HD double h_heat_capacity(const SF3DView &v, uint32_t i, double h, double T)
{
    const double theta = h_theta(v, i, h);
    double hc = (h_bulk_density(h_soil(v, i)) / HC_QUARTZ_DENSITY) * HC_HEAT_CAPACITY_MINERAL + theta * HC_HEAT_CAPACITY_WATER;
    if (v.computeHeatVapor) hc += h_vapor_theta_v(v, i, h, T) * HC_HEAT_CAPACITY_AIR;
    return hc;
}
// getNodeHeatStorage (soilFluxes3D.cpp:1545-1567)
SF3D_HD double h_node_heat_storage(const SF3DView &v, uint32_t i, double h)
{
    const double T = v.T[i], size = v.size[i];
    double heat = h_heat_capacity(v, i, h, T) * size * T;
    if (v.computeHeatVapor) heat += h_vapor_theta_v(v, i, h, T) * h_latent_vaporization(T - HC_ZEROCELSIUS) * HC_WATER_DENSITY * size;
    return heat;
}
// getNodeH_fromTimeSteps (heat.cpp:690-694)
SF3D_HD double h_H_from_steps(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    const double dH = v.H[i] - v.oldH[i];
    return v.oldH[i] + dH * dtHeat / dtWater;
}
SF3D_HD double h_distance3d(const SF3DView &v, uint32_t i, uint32_t j)               // nodeDistance3D, soilPhysics.cpp:331-335
{
    const double dx = v.x[i] - v.x[j], dy = v.y[i] - v.y[j], dz = v.z[i] - v.z[j];
    double n = 0; n += dx * dx; n += dy * dy; n += dz * dz;
    return sqrt(n);
}
// ---- link operands and link factors ------------------------------------------------------------
// Every heat / vapour flux of a link is  coefficient x difference / nodeDistance3D x interfaceArea  with a
// logarithmic mean (Math::computeMean, default type) of a per-node coefficient.  The reference-rounding build
// evaluates exactly that.  Device math (sf3d_view.h) keeps interfaceArea / nodeDistance3D per link (static, one
// load, no division) and every per-node coefficient together with its logarithm (SF3DPair).
SF3D_HD double h_logmean_pre(const SF3DPair a, const SF3DPair b)
{
    // (a - b) / (ln a - ln b).  Nearly equal operands: the series of the logarithmic mean around the arithmetic
    // mean m, x = (a - b) / (a + b):  m (1 - x^2 / 3 - ...), exact to 1e-17 for |x| <= 5e-5, where the difference of
    // two stored logarithms would have lost its digits.  A zero operand (saturated node: no vapour diffusion)
    // gives 0 like the reference's (0 - b) / ln(0 / b).
    if (a.v == b.v) return a.v;
    const double d = a.v - b.v, s = a.v + b.v;
    const bool close = fabs(d) <= 1e-4 * fabs(s);
    const double q = d / (close ? s : (a.l - b.l));
    return close ? 0.5 * s * (1. - q * q * (1. / 3.)) : q;
}
#ifdef SF3D_DEVICE_MATH
SF3D_HD void h_pair_store(double *arr, uint32_t i, double value)
{ SF3DPair p; p.v = value; p.l = log(value); reinterpret_cast<SF3DPair *>(arr)[i] = p; }
SF3D_HD SF3DPair h_pair_load(const double *arr, uint32_t i) { return reinterpret_cast<const SF3DPair *>(arr)[i]; }
SF3D_HD double h_pair_value(const double *arr, uint32_t i) { return reinterpret_cast<const SF3DPair *>(arr)[i].v; }
SF3D_HD double h_pair_mean(const SF3DPair a, const SF3DPair b) { return h_logmean_pre(a, b); }
SF3D_HD double h_link_zeta(const SF3DView &v, uint32_t i, int slot) { return SF3D_LDS(v.ldist3 + (size_t)slot * v.N + i); }
SF3D_HD double h_link_flux(const SF3DView &v, uint32_t i, int slot, double density) { return density * h_link_zeta(v, i, slot); }
SF3D_HD double h_link_store_geometry(double area, double distance3d) { return area / distance3d; }
#else
SF3D_HD void h_pair_store(double *arr, uint32_t i, double value) { arr[i] = value; }
SF3D_HD SF3DPair h_pair_load(const double *arr, uint32_t i) { SF3DPair p; p.v = arr[i]; p.l = 0.; return p; }
SF3D_HD double h_pair_value(const double *arr, uint32_t i) { return arr[i]; }
SF3D_HD double h_pair_mean(const SF3DPair a, const SF3DPair b) { return sf3d_mean(a.v, b.v, 2); }
SF3D_HD double h_link_zeta(const SF3DView &v, uint32_t i, int slot)       // Heat::conduction: area / distance (heat.cpp:647)
{ return v.larea[(size_t)slot * v.N + i] / v.ldist3[(size_t)slot * v.N + i]; }
SF3D_HD double h_link_flux(const SF3DView &v, uint32_t i, int slot, double density)    // ... / distance * area, as written in heat.cpp
{ return density / v.ldist3[(size_t)slot * v.N + i] * v.larea[(size_t)slot * v.N + i]; }
SF3D_HD double h_link_store_geometry(double, double distance3d) { return distance3d; }
#endif
// static heat geometry, filled once per topology: ldist3[slot][i] and hPress[i]
SF3D_HD void sf3d_row_heat_geometry(const SF3DView &v, uint32_t i)
{
    const size_t N = v.N;
    const uint32_t m = v.meta[i];
    v.hPress[i] = h_pressure_from_altitude(v.z[i]);
    for (int slot = 0; slot < SF3D_NLINK; ++slot)
        v.ldist3[(size_t)slot * N + i] = META_HAS_SLOT(m, slot)
            ? h_link_store_geometry(v.larea[(size_t)slot * N + i], h_distance3d(v, i, v.lidx[(size_t)slot * N + i])) : 1.;
}

// getNodeH_fromTimeSteps of a linked node and its sub-step averaged matric head: stored per node by
// sf3d_row_heat_coeffs under device math (same expressions), evaluated on the spot otherwise
SF3D_HD double h_Hs(const SF3DView &v, uint32_t j, double dtHeat, double dtWater)
{
#ifdef SF3D_DEVICE_MATH
    (void)dtHeat; (void)dtWater; return v.hHs[j];
#else
    return h_H_from_steps(v, j, dtHeat, dtWater);
#endif
}
SF3D_HD double h_psi_avg(const SF3DView &v, uint32_t j, double dtHeat, double dtWater)
{
#ifdef SF3D_DEVICE_MATH
    (void)dtHeat; (void)dtWater; return v.hPsiAvg[j];
#else
    return (h_H_from_steps(v, j, dtHeat, dtWater) + v.oldH[j]) * 0.5 - v.z[j];
#endif
}

// linked node of a slot without the dependent 4-byte load of the link index array: from the row's link pattern (kernel
// parameters / the small pattern table) like the sweeps; the explicit matrix column array when patterns are off; the link
// index array on host views
SF3D_HD uint32_t h_link_node(const SF3DView &v, const int32_t *off, uint32_t i, int slot)
{
    if (off || v.mcol) return sf3d_col_index(v, off, i, sf3d_col_of_slot(slot));
    return v.lidx[(size_t)slot * v.N + i];
}

// ---- water-side hooks --------------------------------------------------------------------------
// computeNodeK's vapour term (soilPhysics.cpp:168-169) from the node's current state (bulk potential setter)
SF3D_HD double sf3d_heat_vapor_K(const SF3DView &v, uint32_t i)
{
    const SoilRec &s = h_soil(v, i);
    const double T = h_mean_T(v, i), h = v.H[i] - v.z[i];
    return h_ivk(h_node_ctx(s, T, h, h_theta(v, i, h))) * (HC_GRAVITY / HC_WATER_DENSITY);
}
// One call per soil node and Picard approximation, with the processType::Water arguments (node mean
// temperature, current matric potential; theta from the stored Se, which is the value
// computeNodeTheta_fromSignedPsi recomputes).  Adds the vapour term of computeNodeK
// (soilPhysics.cpp:168-169) to K, stores what the link loop of the assembly reads from both ends of
// every link (mean T, thermal liquid / vapour conductivity) and returns computeNodedThetaVdH
// (soilPhysics.cpp:287-299) through *dThetaVdH when dThetadH is given.
SF3D_HD double sf3d_heat_node_water(const SF3DView &v, uint32_t i, const SoilRec &s, double H, double z, double Se, double K,
                                   const double *dThetadH, double *dThetaVdH)
{
    const double T = h_mean_T(v, i);
    const double h = H - z;
    if (v.computeHeatVapor)
    {
        const double theta = (h >= 0.) ? s.thetaS : sf3d_theta_from_se(s, Se);
        const HeatNodeCtx c = h_node_ctx(s, T, h, theta);
        K += h_ivk(c) * (HC_GRAVITY / HC_WATER_DENSITY);
#ifdef SF3D_DEVICE_MATH
        // the only reader of this pair is the thermal invariant flux of the water rows, which divides the vapour flux by the
        // water density (water.cpp:337): the mean is homogeneous of degree 1, so the division is done once per node here
        // instead of once per link there
        h_pair_store(v.hTVK, i, h_tvk(s, c, v.hPress[i]) * (1. / HC_WATER_DENSITY));
#else
        h_pair_store(v.hTVK, i, h_tvk(s, c, v.hPress[i]));
#endif
        if (dThetadH)
        {
            const double dThetaVdPsi = (c.svc * c.rh / HC_WATER_DENSITY) * ((s.thetaS - theta) * HC_MH2O / (HC_R_GAS * T) - *dThetadH / HC_GRAVITY);
            *dThetaVdH = dThetaVdPsi * HC_GRAVITY;
        }
    }
    v.hTm[i] = T;
    h_pair_store(v.hTLK, i, h_thermal_liquid_conductivity(T - HC_ZEROCELSIUS, h, K));
    return K;
}

// per-node coefficients with the processType::Heat arguments (node temperature, head averaged over the
// heat sub-step): stored by sf3d_row_heat_coeffs before the flux snapshot and before every heat assembly
SF3D_HD void sf3d_row_heat_coeffs(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    const double Hs = h_H_from_steps(v, i, dtHeat, dtWater);
    const double avgH = (Hs + v.oldH[i]) * 0.5 - v.z[i];
#ifdef SF3D_DEVICE_MATH
    v.hHs[i] = Hs; v.hPsiAvg[i] = avgH;         // surface nodes too: the water flux snapshot reads the head of both ends
#endif
    if (i < v.Ns) return;
    const double T = v.T[i];
    const SoilRec &s = h_soil(v, i);
    const HeatNodeCtx c = h_node_ctx(s, T, avgH, h_theta(v, i, avgH));
    const double tvk = h_tvk(s, c, v.hPress[i]);
    h_pair_store(v.hCond, i, h_soil_heat_conductivity(s, c, tvk));
    h_pair_store(v.hIVK, i, h_ivk(c));
    h_pair_store(v.hTVK, i, tvk);
    // computeThermalLiquidFlux, processType::Heat (heat.cpp:458-500): its head is the sub-step average only
    // when the heat step differs from the water step
    const double liquidH = (dtHeat != dtWater) ? avgH : (v.H[i] + v.oldH[i]) * 0.5 - v.z[i];
    h_pair_store(v.hTLKh, i, h_thermal_liquid_conductivity(T - HC_ZEROCELSIUS, liquidH, v.K[i]));
}

// computeThermalLiquidFlux / computeThermalVaporFlux (heat.cpp:458-553), processType::Heat branch: node
// temperatures, conductivities stored per node by sf3d_row_heat_coeffs with exactly these arguments
SF3D_HD double h_thermal_liquid_flux_heat(const SF3DView &v, uint32_t i, int slot, uint32_t j)
{
    const double avg = h_pair_mean(h_pair_load(v.hTLKh, i), h_pair_load(v.hTLKh, j));     // computeMean default = Logarithmic
    return h_link_flux(v, i, slot, avg * (v.T[j] - v.T[i]));
}
SF3D_HD double h_thermal_vapor_flux_heat(const SF3DView &v, uint32_t i, int slot, uint32_t j, double dtHeat, double dtWater, bool usePre)
{
    double avg;
    if (usePre) avg = h_pair_mean(h_pair_load(v.hTVK, i), h_pair_load(v.hTVK, j));
    else
    {
        // after the heat solve (saveNodeHeatFluxes): the conductivities of the NEW temperatures, evaluated on the spot
        const double srcH = h_psi_avg(v, i, dtHeat, dtWater);
        const double dstH = h_psi_avg(v, j, dtHeat, dtWater);
        const double a = h_thermal_vapor_conductivity(v, i, v.T[i], srcH);
        const double b = h_thermal_vapor_conductivity(v, j, v.T[j], dstH);
        avg = sf3d_mean(a, b, 2);
    }
    return h_link_flux(v, i, slot, avg * (v.T[j] - v.T[i]));
}
// water.cpp:329-340: thermal liquid (+ vapour / rho_w) flux added to the row's invariant fluxes
// (processType::Water branch).  tl / tv / tm: thermal liquid conductivity, thermal vapour conductivity
// and mean temperature of the two ends, stored by sf3d_heat_node_water.
SF3D_HD double sf3d_heat_thermal_invariant(const SF3DView &v, uint32_t i, int slot, const SF3DPair tli, const SF3DPair tvi, double tmi,
                                          const SF3DPair tlj, const SF3DPair tvj, double tmj)
{
    const double dT = tmj - tmi;
#ifdef SF3D_DEVICE_MATH
    const double zeta = h_link_zeta(v, i, slot);                // one load for both fluxes; tv pairs are stored / rho_w
    double f = (h_pair_mean(tli, tlj) * dT) * zeta;
    if (v.computeHeatVapor) f += (h_pair_mean(tvi, tvj) * dT) * zeta;
    return f;
#else
    double f = h_link_flux(v, i, slot, h_pair_mean(tli, tlj) * dT);
    if (v.computeHeatVapor) f += h_link_flux(v, i, slot, h_pair_mean(tvi, tvj) * dT) / HC_WATER_DENSITY;
    return f;
#endif
}

// one soil row's invariant fluxes of the water system: thermal liquid (+ thermal vapour / rho_w) flux of every
// soil-soil link, accumulated in the reference's link order (Up, Lateral 0..7, Down: computeLinearSystemElement,
// cpusolver.cpp:352-374, through computeLinkFluxes, water.cpp:329-340).  Operands were stored by the node phase.
SF3D_HD void sf3d_row_thermal_invariant(const SF3DView &v, uint32_t i)
{
    if (i < v.Ns) return;
    const int32_t *off = sf3d_row_pattern(v, i);
#ifdef SF3D_DEVICE_MATH
    // Two passes over the links, one per conductivity (liquid, then vapour): each keeps ONE operand pair per link end live.
    // The single-pass form spilled at the 32 registers this kernel runs best with (ncu: 12 % of the stall samples on the
    // spill stores, LSU throttling on top); the second pass re-reads the linked temperatures and the link geometry from L1.
    // The sum is taken liquid links first, then vapour links (a rounding-level reordering of the reference's per-link sums).
    const double tmi = v.hTm[i];
    double invariant = 0.;
    const int nPass = v.computeHeatVapor ? 2 : 1;
    for (int pass = 0; pass < nPass; ++pass)
    {
        const double *op = pass ? v.hTVK : v.hTLK;              // vapour pairs are stored / rho_w (sf3d_heat_node_water)
        const SF3DPair ai = h_pair_load(op, i);
        #pragma unroll kThermalUnroll
        for (int c = 0; c < SF3D_NLINK; ++c)
        {
            const uint32_t j = sf3d_col_index(v, off, i, c);
            if (j == i || j < v.Ns) continue;                   // absent link, or the infiltration link of the first soil layer
            const double zeta = h_link_zeta(v, i, sf3d_slot_of_col(c));
            invariant += (h_pair_mean(ai, h_pair_load(op, j)) * (v.hTm[j] - tmi)) * zeta;
        }
    }
    v.hInv[i] = invariant;
#else
    const SF3DPair tli = h_pair_load(v.hTLK, i);
    SF3DPair tvi = {0., 0.};
    if (v.computeHeatVapor) tvi = h_pair_load(v.hTVK, i);
    const double tmi = v.hTm[i];
    double invariant = 0.;
    #pragma unroll kThermalUnroll
    for (int c = 0; c < SF3D_NLINK; ++c)
    {
        const uint32_t j = sf3d_col_index(v, off, i, c);
        if (j == i || j < v.Ns) continue;                   // absent link, or the infiltration link of the first soil layer
        SF3DPair tvj = {0., 0.};
        if (v.computeHeatVapor) tvj = h_pair_load(v.hTVK, j);
        invariant += sf3d_heat_thermal_invariant(v, i, sf3d_slot_of_col(c), tli, tvi, tmi, h_pair_load(v.hTLK, j), tvj, v.hTm[j]);
    }
    v.hInv[i] = invariant;
#endif
}

// computeNodeAtmosphericLatentVaporFlux (heat.cpp:988-1007), node = HeatSurface soil node
SF3D_HD double h_atmospheric_latent_vapor_flux(const SF3DView &v, uint32_t i)
{
    const uint32_t up = v.lidx[i];
    if (!(up < v.Ns)) return 0.;
    const double satP = h_sat_vapor_pressure(v.hbT[i] - HC_ZEROCELSIUS);
    const double satC = h_vapor_conc_from_pressure(satP, v.hbT[i]);
    const double boundaryVapor = satC * (v.hbRH[i] / 100.);
    const double deltaVapor = boundaryVapor - h_vapor_from_psi_temp(v.H[i] - v.z[i], v.T[i]);     // getNodeVapor
    const double total = 1. / ((1. / v.hbAero[i]) + (1. / v.hbSoilCond[i]));
    return deltaVapor * total;
}
// computeNodeAtmosphericLatentSurfaceWaterFlux (heat.cpp:1013-1036), node = surface node, down = HeatSurface node
SF3D_HD double h_atmospheric_surface_water_flux(const SF3DView &v, uint32_t down)
{
    const double satP = h_sat_vapor_pressure(v.hbT[down] - HC_ZEROCELSIUS);
    const double satC = h_vapor_conc_from_pressure(satP, v.hbT[down]);
    const double boundaryVapor = satC * (v.hbRH[down] / 100.);
    const double deltaVapor = boundaryVapor - satC;
    return deltaVapor * v.hbAero[down];
}
// getNodeSurfaceWaterFraction (soilPhysics.cpp:313-323)
SF3D_HD double h_surface_water_fraction(const SF3DView &v, uint32_t s)
{
    if (!(s < v.Ns)) return 0.;
    const double hV = sf3d_max(0., v.H[s] - v.z[s]);
    const double h0 = sf3d_max(0.001, v.pond[s]);
    return sf3d_min(1., hV / h0);
}

// HeatSurface branch of updateBoundaryWaterData (water.cpp:708-747), soil-node side: soil evaporation
SF3D_HD double sf3d_heat_surface_boundary(const SF3DView &v, uint32_t i, double dt, double *)
{
    const uint32_t m = v.meta[i];
    const bool upLinked = META_HAS_SLOT(m, 0);
    const uint32_t up = upLinked ? v.lidx[i] : 0xFFFFFFFFu;
    const double fraction = upLinked ? h_surface_water_fraction(v, up) : 0.;
    const double area = v.larea[i];
    double soilEvap = h_atmospheric_latent_vapor_flux(v, i) / HC_WATER_DENSITY * area;
    if (fraction > 0.) soilEvap *= (1. - fraction);
    const SoilRec &s = h_soil(v, i);
    const double thetaV = sf3d_theta_from_se(s, v.Se[i]);
    soilEvap = (soilEvap < 0.) ? sf3d_max(soilEvap, -(thetaV - s.thetaR) * v.size[i] / dt)
                               : sf3d_min(soilEvap, (s.thetaS - s.thetaR) * v.size[i] / dt);
    return soilEvap;
}
// the same branch, surface-node side (the reference writes the up node from the soil node's
// iteration, water.cpp:722-736; here the surface node pulls it through its Down link: Q9).
// Returns the surface-water evaporation [m3 s-1]; *active = 0 when nothing is to be applied.
SF3D_HD double sf3d_heat_surface_pull(const SF3DView &v, uint32_t i, double dt, int *active)
{
    *active = 0;
    const uint32_t m = v.meta[i];
    if (!META_HAS_SLOT(m, 1)) return 0.;
    const uint32_t down = v.lidx[(size_t)v.N + i];
    if (META_BT(v.meta[down]) != BT_HEAT_SURFACE) return 0.;
    if (!META_HAS_SLOT(v.meta[down], 0) || v.lidx[down] != i) return 0.;
    const double fraction = h_surface_water_fraction(v, i);
    if (!(fraction > 0.)) return 0.;
    const double area = v.larea[down];                            // linkData[0].interfaceArea of the soil node
    double surfEvap = h_atmospheric_surface_water_flux(v, down) / HC_WATER_DENSITY * area;
    surfEvap *= fraction;
    const double waterVolume = (v.H[i] - v.z[i]) * v.size[i];
    surfEvap = sf3d_max(surfEvap, -waterVolume / dt);
    *active = 1;
    return surfEvap;
}

// ==========================================================================================
// Heat::updateConductance per node (heat.cpp:214-235) with computeNodeAerodynamicConductance
// (heat.cpp:882-951, fixed-point iteration, at most 100 rounds)
// ==========================================================================================
SF3D_HD double h_aerodynamic_conductance(const SF3DView &v, uint32_t i)
{
    const double heightT = v.hbHeightT[i], heightWind = v.hbHeightWind[i];
    const double soilT = v.T[i], rHeight = v.hbRough[i], airT = v.hbT[i];
    const double wind = sf3d_max(v.hbWind[i], 0.01);
    const double zeroPlane = 0.77 * rHeight;
    const double rMomentum = 0.13 * rHeight;
    const double rHeat = 0.2 * rMomentum;
    double psiM = 0., psiH = 0.;
    const double cH = h_air_vol_specific_heat(h_pressure_from_altitude(heightWind), airT);
    bool first = true;
    double oldHf = SF3D_NODATA, K = SF3D_NODATA;
    for (int counter = 0; counter < 100; ++counter)
    {
        const double uStar = HC_VON_KARMAN * wind / (log((heightWind - zeroPlane + rMomentum) / rMomentum) + psiM);
        K = HC_VON_KARMAN * uStar / (log((heightT - zeroPlane + rHeat) / rHeat) + psiH);
        const double Hf = K * cH * (soilT - airT);
        const double sP = -HC_VON_KARMAN * heightWind * HC_GRAVITY * Hf / (cH * airT * (h_pow3(uStar)));
        if (sP > 0) { psiH = 6 * log(1 + sP); psiM = psiH; }
        else { psiH = -2 * log((1 + sqrt(1 - 16 * sP)) / 2); psiM = 0.6 * psiH; }
        if (first) first = false;
        else if (fabs(Hf - oldHf) < 0.01) break;
        oldHf = Hf;
    }
    return K;
}
SF3D_HD void sf3d_row_update_conductance(const SF3DView &v, uint32_t i)
{
    if (META_BT(v.meta[i]) != BT_HEAT_SURFACE) return;
    v.hbAero[i] = h_aerodynamic_conductance(v, i);
    const double theta = h_theta(v, i, v.H[i] - v.z[i]);
    v.hbSoilCond[i] = 1. / h_soil_surface_resistance(theta);
}

// ==========================================================================================
// Heat::saveNodeWaterFluxes (heat.cpp:109-138): per link water / vapour flux snapshot, float-rounded
// ==========================================================================================
SF3D_HD double h_isothermal_vapor_flux(const SF3DView &v, uint32_t i, int slot, uint32_t j, double dtHeat, double dtWater)   // :561-582
{
    const double srcH = h_psi_avg(v, i, dtHeat, dtWater);
    const double dstH = h_psi_avg(v, j, dtHeat, dtWater);
    // operands = computeNodeIsothermalVaporConductivity(node, T[node], its averaged head), see sf3d_row_heat_coeffs
    const double avg = h_pair_mean(h_pair_load(v.hIVK, i), h_pair_load(v.hIVK, j));
    const double srcPsi = srcH * HC_GRAVITY, dstPsi = dstH * HC_GRAVITY;
    const double deltaPsi = dstPsi - srcPsi;
    return h_link_flux(v, i, slot, avg * deltaPsi);
}
SF3D_HD void sf3d_row_save_water_fluxes(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    const size_t N = v.N;
    const uint32_t m = v.meta[i];
    const int32_t *off = sf3d_row_pattern(v, i);
    #pragma unroll kHeatLinkUnroll
    for (int slot = 0; slot < SF3D_NLINK; ++slot)
    {
        if (!META_HAS_SLOT(m, slot)) continue;
        const size_t li = (size_t)slot * N + i;
        const uint32_t j = h_link_node(v, off, i, slot);
        const double srcAvgH = h_Hs(v, i, dtHeat, dtWater);
        const double dstAvgH = h_Hs(v, j, dtHeat, dtWater);
        const double A = v.mval[(size_t)sf3d_col_of_slot(slot) * N + i];      // normalised entry x 1.0 (Q1); 0 if not stored (Q2)
        const double isoLiquid = A * (srcAvgH - dstAvgH);
        const bool deep = !(i < v.Ns) && !(j < v.Ns);
        const double isoVapor = deep ? h_isothermal_vapor_flux(v, i, slot, j, dtHeat, dtWater) : 0.;
        const double thLiquid = deep ? h_thermal_liquid_flux_heat(v, i, slot, j) : 0.;
        const double thVapor = deep ? h_thermal_vapor_flux_heat(v, i, slot, j, dtHeat, dtWater, true) : 0.;
        v.lwFlux[li] = (double)(float)(isoLiquid - isoVapor / HC_WATER_DENSITY + thLiquid);
        v.lvFlux[li] = (double)(float)(isoVapor + thVapor);
        if (v.hfSaveMode == 2)
        {
            v.lfluxes[(size_t)5 * SF3D_NLINK * N + li] = (double)(float)isoLiquid;
            v.lfluxes[(size_t)6 * SF3D_NLINK * N + li] = (double)(float)thLiquid;
            v.lfluxes[(size_t)7 * SF3D_NLINK * N + li] = (double)(float)isoVapor;
            v.lfluxes[(size_t)8 * SF3D_NLINK * N + li] = (double)(float)thVapor;
        }
    }
}

// ==========================================================================================
// Heat::updateBoundaryHeatData per node (heat.cpp:243-320); returns the node's Courant value
// ==========================================================================================
SF3D_HD double sf3d_row_boundary_heat(const SF3DView &v, uint32_t i, double maxTimeStep)
{
    if (i < v.Ns) return 0.;
    double flux = v.hSink[i];
    const uint32_t bt = META_BT(v.meta[i]);
    double courant = 0.;
    if (bt == BT_NONE) { v.hFlux[i] = flux; return 0.; }
    const double upArea = v.larea[i];
    if (bt == BT_HEAT_SURFACE)
    {
        double adv = 0., sens = 0., lat = 0., rad = 0.;
        if (v.hbNetIrr[i] != SF3D_NODATA) rad = v.hbNetIrr[i];
        // computeNodeAtmosphericSensibleHeatFlux (heat.cpp:957-968)
        {
            const uint32_t up = v.lidx[i];
            if (up < v.Ns)
            {
                const double pressure = v.hPress[i];
                const double deltaT = v.hbT[i] - v.T[i];
                sens += h_air_vol_specific_heat(pressure, v.hbT[i]) * deltaT * v.hbAero[i];
            }
        }
        if (v.computeHeatVapor)
        {
            // computeNodeAtmosphericLatentHeatFlux (heat.cpp:974-982) / upLinkArea
            const uint32_t up = v.lidx[i];
            double latent = 0.;
            if (up < v.Ns) latent = v.bRate[i] * HC_WATER_DENSITY * h_latent_vaporization(v.T[i] - HC_ZEROCELSIUS);
            lat += latent / upArea;
        }
        if (v.computeHeatAdvection)
        {
            double advT = v.hbT[i];
            const double wFlux = v.lwFlux[i];                       // Up link water flux
            if (wFlux > 0.) adv = wFlux * HC_HEAT_CAPACITY_WATER * advT / upArea;
            if (v.bRate[i] < 0.) advT = v.T[i];
            adv += v.bRate[i] * HC_WATER_DENSITY * HC_HEAT_CAPACITY_WATER_VAPOR * advT / upArea;
        }
        v.hbAdv[i] = adv; v.hbSens[i] = sens; v.hbLat[i] = lat; v.hbRad[i] = rad;
        flux += upArea * (rad + sens + lat + adv);
        const double hc = h_heat_capacity(v, i, v.oldH[i], v.oldT[i]);      // (sic) oldPressureHead passed as h, heat.cpp:293
        courant = fabs(flux) * maxTimeStep / (hc * v.size[i]);
    }
    else if (bt == BT_FREE_DRAINAGE || bt == BT_PRESCRIBED)
    {
        if (v.computeHeatAdvection)
        {
            const double wFlux = v.bRate[i];
            const double advT = (wFlux < 0) ? v.T[i] : v.hbFixT[i];
            const double adv = wFlux * HC_HEAT_CAPACITY_WATER * advT / upArea;
            v.hbAdv[i] = adv;
            flux += upArea * adv;
        }
        if (v.hbFixT[i] != SF3D_NODATA)
        {
            const double avgH = (v.H[i] + v.oldH[i]) * 0.5;
            const double bK = h_soil_heat_conductivity(v, i, v.T[i], avgH - v.z[i]);
            const double deltaT = v.hbFixT[i] - v.T[i];
            flux += bK * deltaT / v.hbFixDepth[i] * upArea;
        }
    }
    v.hFlux[i] = flux;
    return courant;
}

// ==========================================================================================
// CPUSolver::heatLoop, per-node pieces (cpusolver.cpp:471-605)
// ==========================================================================================
// x = T ; oldT = T ; C = heat capacity x volume  (:476-491)
SF3D_HD void sf3d_row_heat_begin(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    const double T = v.T[i];
    v.x0[i] = T;
    v.oldT[i] = T;
    if (i < v.Ns) return;
    const double nodeH = h_H_from_steps(v, i, dtHeat, dtWater);
    const double avgH = (v.oldH[i] + nodeH) * 0.5 - v.z[i];
    v.cap[i] = h_heat_capacity(v, i, avgH, T) * v.size[i];
}

// saveNodeHeatSpecificFlux (heat.cpp:198-212): float-rounded accumulation into HeatTotal
SF3D_HD void h_save_specific_flux(const SF3DView &v, uint32_t i, int slot, int type, double value)
{
    if (v.hfSaveMode == 0) return;
    const size_t N = v.N, li = (size_t)slot * N + i;
    value = (double)(float)value;
    double &total = v.lfluxes[li];                              // type 0 = HeatTotal
    total = (double)(float)((total == SF3D_NODATA) ? value : total + value);
    if (v.hfSaveMode == 2) v.lfluxes[(size_t)type * SF3D_NLINK * N + li] = value;
}

// Heat::conduction (heat.cpp:643-661)
SF3D_HD double h_conduction(const SF3DView &v, uint32_t i, int slot, uint32_t j, double dtHeat, double dtWater)
{
    const double zeta = h_link_zeta(v, i, slot);
    (void)dtHeat; (void)dtWater;
    // operands = computeNodeHeatSoilConductivity(node, T[node], its averaged head), see sf3d_row_heat_coeffs
    return zeta * h_pair_mean(h_pair_load(v.hCond, i), h_pair_load(v.hCond, j));
}
// computeAdvectiveFlux (heat.cpp:606-621)
SF3D_HD double h_advective_flux(const SF3DView &v, uint32_t i, int slot, uint32_t j)
{
    const size_t li = (size_t)slot * v.N + i;
    const double lw = v.lwFlux[li];
    const double lT = v.T[(lw < 0.) ? i : j];
    const double vw = v.lvFlux[li];
    const double vT = v.T[(vw < 0.) ? i : j];
    return (HC_HEAT_CAPACITY_WATER * lw) * lT + (HC_HEAT_CAPACITY_WATER_VAPOR * vw) * vT;
}

// one row of the heat system (cpusolver.cpp:496-568).  Column order Up, Down, Lateral 0..7
// (cpusolver.cpp:524-540, SURVEY Q3); stored in SLOT order, which is the same order.
SF3D_HD void sf3d_row_heat_assemble(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    const size_t N = v.N;
    // save mode Total: this pass writes the HeatTotal slot of EVERY link (the value or NODATA), which is the reset of
    // resetFluxValues(true, false) (heat.cpp:55-78) and the first saveNodeHeatSpecificFlux in one store, without a read
    const bool totalOnly = v.hfSaveMode == 1;
    if (i < v.Ns)
    {
        #pragma unroll 1
        for (int s = 0; s < SF3D_NLINK; ++s)
        {
            v.mval[(size_t)s * N + i] = 0.;
            if (totalOnly) v.lfluxes[(size_t)s * N + i] = SF3D_NODATA;
        }
        v.hdiag[i] = 0.;
        v.b[i] = v.T[i];
        return;
    }
    const uint32_t m = v.meta[i];
    const double nodeT = v.T[i];
    const double nodeH = h_H_from_steps(v, i, dtHeat, dtWater);
    const double oldPsi = v.oldH[i] - v.z[i];
    const SoilRec &s = h_soil(v, i);
    // the two water contents are evaluated once and shared by the liquid and the vapour terms (the reference
    // evaluates computeNodeTheta_fromSignedPsi with the same arguments inside computeNodeVaporThetaV again).
    // theta(oldPsi): Se of the step's starting head is the stored SeOld, the value computeNodeSe_fromPsi returns
    // for |oldPsi| (same function, same argument: sf3d_row_begin_try)
    const double thetaNew = sf3d_theta_from_signed_psi(s, v.wrcModel, nodeH - v.z[i]);
    const double thetaOld = (oldPsi >= 0.) ? s.thetaS : sf3d_theta_from_se(s, v.SeOld[i]);
    const double dTheta = thetaNew - thetaOld;
    double heatCapacity = dTheta * HC_HEAT_CAPACITY_WATER * nodeT;
    if (v.computeHeatVapor)
    {
        // computeNodeVaporThetaV (heat.cpp:868-875) with the water contents above
        const double vNew = h_vapor_from_psi_temp(nodeH - v.z[i], nodeT) / HC_WATER_DENSITY * (s.thetaS - thetaNew);
        const double vOld = h_vapor_from_psi_temp(oldPsi, v.oldT[i]) / HC_WATER_DENSITY * (s.thetaS - thetaOld);
        const double dThetaV = vNew - vOld;
        heatCapacity += dThetaV * HC_HEAT_CAPACITY_AIR * nodeT;
        heatCapacity += dThetaV * h_latent_vaporization(nodeT - HC_ZEROCELSIUS) * HC_WATER_DENSITY;
    }
    heatCapacity *= v.size[i];

    const double wf = v.heatWF;
    double sumDP = 0., sumF0 = 0., invariant = 0.;
    double val[SF3D_NLINK];
    const int32_t *off = sf3d_row_pattern(v, i);
    #pragma unroll kHeatLinkUnroll
    for (int slot = 0; slot < SF3D_NLINK; ++slot)
    {
        val[slot] = 0.;
        const uint32_t j = META_HAS_SLOT(m, slot) ? h_link_node(v, off, i, slot) : 0u;
        if (!META_HAS_SLOT(m, slot) || j < v.Ns)                    // absent link / !isHeatNode(linked), heat.cpp:423
        {
            if (totalOnly) v.lfluxes[(size_t)slot * N + i] = SF3D_NODATA;
            continue;
        }
        const double e = h_conduction(v, i, slot, j, dtHeat, dtWater);
        double latent = 0., advective = 0.;
        double total = SF3D_NODATA;                                 // saveNodeHeatSpecificFlux on a freshly reset slot
        if (v.computeHeatVapor)
        {
            // computeIsothermalLatentHeatFlux (heat.cpp:590-600)
            const double avgLambda = (h_latent_vaporization(v.T[i] - HC_ZEROCELSIUS) + h_latent_vaporization(v.T[j] - HC_ZEROCELSIUS)) * 0.5;
            latent = avgLambda * h_isothermal_vapor_flux(v, i, slot, j, dtHeat, dtWater);
            if (totalOnly) total = (double)(float)latent;
            else h_save_specific_flux(v, i, slot, 2, latent);
        }
        if (v.computeHeatAdvection)
        {
            advective = h_advective_flux(v, i, slot, j);
            if (totalOnly)
            {
                const double a = (double)(float)advective;
                total = (double)(float)((total == SF3D_NODATA) ? a : total + a);
            }
            else h_save_specific_flux(v, i, slot, 4, advective);
        }
        if (totalOnly) v.lfluxes[(size_t)slot * N + i] = total;
        invariant += advective + latent;
        // cpusolver.cpp:545-552
        sumDP += e * wf;
        const double dT0 = v.oldT[j] - v.oldT[i];
        sumF0 += e * (1. - wf) * dT0;
        val[slot] = e * (-wf);
    }
    const double capOverDt = v.cap[i] / dtHeat;
    const double diag = sumDP + capOverDt;
    double b = v.cap[i] * v.oldT[i] / dtHeat - heatCapacity / dtHeat + v.hFlux[i] + invariant + sumF0;
    if (diag > 0)
    {
#ifdef SF3D_DEVICE_MATH
        const double inv = 1. / diag;                   // one division per row instead of eleven
        b *= inv;
        #pragma unroll 1
        for (int slot = 0; slot < SF3D_NLINK; ++slot) val[slot] *= inv;
#else
        b /= diag;
        #pragma unroll 1
        for (int slot = 0; slot < SF3D_NLINK; ++slot) val[slot] /= diag;
#endif
    }
    #pragma unroll 1
    for (int slot = 0; slot < SF3D_NLINK; ++slot) v.mval[(size_t)slot * N + i] = val[slot];
    v.hdiag[i] = diag;
    v.b[i] = b;
}

// one Jacobi row of the heat system; returns |dx| (the reference sweeps Gauss-Seidel in place with
// the same row formula and an infinity norm, heat.cpp:664-685; see DESIGN.md, Q6).  Entries are stored and
// summed in SLOT order (= the reference's column order Up, Down, Lateral 0..7); the linked node of a slot comes
// from sf3d_row_cols like in the water sweep (absent links and links to surface nodes hold a zero entry pointing at
// the row itself / at a finite x), so no meta word is read.
SF3D_HD double sf3d_row_heat_jacobi(const SF3DView &v, uint32_t i, const double *__restrict__ xin, double *__restrict__ xout,
                                    double *xnewOut = nullptr)
{
    const size_t N = v.N;
    const double xold = xin[i];
    if (xnewOut) *xnewOut = xold;
    if (i < v.Ns || SF3D_LDS(v.hdiag + i) == 0.) { xout[i] = xold; return 0.; }
    uint32_t j[SF3D_NLINK];
    sf3d_row_cols(v, i, j);                     // j[c]: COLUMN order (Up, Lateral 0..7, Down)
    double xnew = SF3D_LDS(v.b + i);
    #pragma unroll
    for (int slot = 0; slot < SF3D_NLINK; ++slot)
    {
        const double A = SF3D_LDS(v.mval + (size_t)slot * N + i);
        xnew -= A * xin[j[sf3d_col_of_slot(slot)]];
    }
    xout[i] = xnew;
    if (xnewOut) *xnewOut = xnew;
    return fabs(xnew - xold);
}

// T = x ; heat storage and sink sums (cpusolver.cpp:573-577, heat.cpp:342-370)
SF3D_HD void sf3d_row_heat_post(const SF3DView &v, uint32_t i, const double *__restrict__ x, double dtHeat, double dtWater,
                               int mode, double *storage, double *sinkSum)
{
    *storage = 0.; *sinkSum = 0.;
    if (i < v.Ns) return;
    if (mode == 0) v.T[i] = x[i];
    const double nodeH = (mode == 2) ? v.H[i] : h_H_from_steps(v, i, dtHeat, dtWater);
    *storage = h_node_heat_storage(v, i, nodeH - v.z[i]);
    const double f = v.hFlux[i];
    *sinkSum = (f != 0.) ? f * dtHeat : 0.;
}

// saveNodeHeatFluxes (heat.cpp:160-196) + oldT = T (cpusolver.cpp:598-602)
SF3D_HD void sf3d_row_heat_accept(const SF3DView &v, uint32_t i, double dtHeat, double dtWater)
{
    if (i < v.Ns) return;
    const size_t N = v.N;
    if (v.hfSaveMode != 0)
    {
        const uint32_t m = v.meta[i];
        const int32_t *off = sf3d_row_pattern(v, i);
        #pragma unroll kHeatAcceptUnroll
        for (int slot = 0; slot < SF3D_NLINK; ++slot)
        {
            if (!META_HAS_SLOT(m, slot)) continue;
            const uint32_t j = h_link_node(v, off, i, slot);
            if (j < v.Ns) continue;
            const double mv = v.mval[(size_t)slot * N + i] * v.hdiag[i];     // getMatrixElement: value x diagonal (kept for heat)
            double heatDiff = mv * (v.T[i] - v.T[j]) * v.heatWF + mv * (v.oldT[i] - v.oldT[j]) * (1. - v.heatWF);
            if (v.hfSaveMode == 1) h_save_specific_flux(v, i, slot, 0, heatDiff);
            else
            {
                if (v.computeHeatVapor)
                {
                    const double thLatent = h_thermal_vapor_flux_heat(v, i, slot, j, dtHeat, dtWater, false) * h_latent_vaporization(v.T[i] - HC_ZEROCELSIUS);
                    h_save_specific_flux(v, i, slot, 3, thLatent);
                    heatDiff -= thLatent;
                }
                h_save_specific_flux(v, i, slot, 1, heatDiff);
            }
        }
    }
}
