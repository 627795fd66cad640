// sb2_ptgsk.cuh -- the pt_gs_k cell stack on sm_100a: a three-kernel phase pipeline per time window
// (forcing terms -> gamma_snow -> response, see "the phase pipeline" below).
//
// One thread per cell in the two stateful kernels, the fp64 state values in registers for the whole time window, forcing,
// scratch and collected series laid out [time][cell] so each step's loads and stores are coalesced 8-byte accesses,
// per-catchment discharge reduced by a segmented warp shuffle into fixed slots (deterministic).
//
// Follows, step for step:
//   run_pt_gs_k                      core/pt_gs_k.h:340-397
//   gamma_snow::calculator::step     core/gamma_snow.h:291-493 (+ calc_snow_state :230-260, corr_lwc :214-227,
//                                    reset_snow_pack :262-274, calc_q :209-212)
//   kirchner::calculator::step       core/kirchner.h:213-235 over odeint's controlled dopri5 dense output
//   priestley_taylor                 core/priestley_taylor.h:75-103
//   actual_evapotranspiration        core/actual_evapotranspiration.h:40-62
//   glacier_melt::step               core/glacier_melt.h:47-52
//   collectors                       core/pt_gs_k_cell_model.h:81-90,116-123,193-205
#pragma once
#include <stdint.h>

#include "sb2_math.cuh"

// Every device function of this file reads the exp / log tables from the block's shared memory (sb_*<true>): a kernel that calls
// into it starts with sb_math_stage_tables() and is launched with SB2_MTAB_BYTES of dynamic shared memory.
namespace sb2 {

// parameter set as the kernel reads it (host fills it from parameter::set order, core/pt_gs_k.h:77-112)
struct PtgskParam {
    double c1, c2, c3;            // kirchner
    double ae_scale_factor;       // ae
    double tx, wind_scale, max_water, wind_const, fast_albedo_decay_rate, slow_albedo_decay_rate, surface_magnitude, max_albedo,
        min_albedo, snowfall_reset_depth, snow_cv, glacier_albedo;  // gs
    double p_corr_scale_factor;
    double snow_cv_forest_factor, snow_cv_altitude_factor;
    double pt_albedo, pt_alpha;
    double initial_bare_ground_fraction;
    double gm_dtf, gm_direct_response;
    double reservoir_direct_response_fraction;
    // per-run constants the reference recomputes every step from p and dt (gamma_snow.h:341-343), evaluated once on the host
    double slow_albedo_decay_step;  // 0.5*albedo_range*dt_in_days/slow_albedo_decay_rate
    double fast_albedo_decay_step;  // pow(2.0, -dt_in_days/fast_albedo_decay_rate)
    int32_t winter_end_day_of_year;
    int32_t n_winter_days;
    int32_t calculate_iso_pot_energy;
    int32_t pad_;
    // divisors that depend on the parameter set only, with their reciprocals (div_by, sb2_math.cuh): snowfall_reset_depth,
    // 1 - initial_bare_ground_fraction, max_water, ae_scale_factor
    InvDivisor inv_snowfall_reset_depth, inv_one_minus_y0, inv_max_water, inv_ae_scale;
};

// device error bits.  gamma_snow's "Mass balance violation" (gamma_snow.h:310-311) has none: with snow, rain = prec, 0 or 0, prec the tested
// |snow + rain - prec| is 0, or NaN for a non-finite prec, and neither exceeds 1e-8 -- the throw is unreachable.
enum : int { ERR_KIRCHNER_STEP = 1 };

struct PtgskRunArgs {
    int64_t n_cells;
    // static per-cell data (SoA)
    const double* __restrict__ z;
    const double* __restrict__ area;
    const double* __restrict__ glacier;
    const double* __restrict__ lake;
    const double* __restrict__ reservoir;
    const double* __restrict__ forest;
    const int32_t* __restrict__ pset;          // parameter-set index per cell
    const uint8_t* __restrict__ active;        // catchment calculation filter expanded per cell (nullable = all)
    const PtgskParam* __restrict__ params;
    double* __restrict__ state;                // [9][n_cells]
    // forcing window: element (local step i, cell c) of variable v at f[v][i*n_cells + c]
    const double* __restrict__ f[5];
    // time
    int n_steps;                               // steps in this launch
    int64_t first_step;                        // absolute index on the model axis of local step 0
    double dt_seconds;                         // to_seconds(dt)
    double dt_hours;                           // to_seconds(T1-T0)/to_seconds(deltahours(1))
    double dt_us;                              // double(dt.count())
    double bb0;                                // 0.98*sigma*pow(273.15,4), gamma_snow.h:286 (host-evaluated)
    InvDivisor inv_dt_seconds, inv_dt_us;      // the step length as a divisor (div_by, sb2_math.cuh)
    double dtb[26];                            // dt_hours * (Dormand-Prince tableau entry k), host-evaluated: the first try of every Kirchner step
    // the region parameter set (params[0]) by value: with no catchment overrides and no ensemble every cell reads its parameters from
    // the kernel's constant bank (UPAR kernels) instead of through a pointer the step's stores might alias
    PtgskParam par0;
    // [T] x = calendar::day_of_year(period.start), y = (period.start - trim(period.start, YEAR)) in seconds, UTC: one 8-byte load per step
    const int2* __restrict__ day_sec_of_year;
    // collected series: element (absolute step - out_first_step, cell) at r[s][...*n_cells + c]; null = not collected
    double* __restrict__ resp[8];
    double* __restrict__ st[9];
    int64_t out_first_step;                    // absolute step stored at row 0 of resp/st
    int collect_end_state;                     // write the T+1'th state point after the last step
    // catchment partial sums: slot of each cell's (warp, catchment-run) segment, head flag; partial[i][slot][2]
    const int32_t* __restrict__ slot;
    double* __restrict__ partial;
    int64_t n_slots;
    int* __restrict__ error_flag;
    // parameter-set ensemble (calibration): blockIdx.y = member; member e steps its own state / partial sums with the
    // region parameter replaced by ens_params[e] (cells with a catchment override keep it, model_calibration.h:830-832)
    const PtgskParam* __restrict__ ens_params;  // null = no ensemble
    int64_t ens_state_stride, ens_partial_stride;
    // phase pipeline scratch, element (local step i, cell c) at scr[k][i*n_cells + c]:
    // 0 potential evapotranspiration [mm/h], 1 long-wave addend, 2 turbulent addend, 3 snow outflow [mm/h], 4 snow covered area
    double* __restrict__ scr[5];
    int64_t ens_scr_stride;  // elements between two members' scratch arrays
    // time split of the snow / response kernels (step_slice_begin): steps per work unit (0 = one unit per cell group), ticket counter per
    // ensemble member, finished units per (member, cell group)
    int unit_steps;
    int* __restrict__ tickets;
    int* __restrict__ progress;
};
enum : int { SCR_POT = 0, SCR_LW = 1, SCR_TADD = 2, SCR_OUTFLOW = 3, SCR_SCA = 4 };

#define SB2_BLOCK 32       // threads per block of the hbv step kernel (sb2_hbv.cuh)

struct GsState { double albedo, lwc, surface_heat, alpha, sdc_melt_mean, acc_melt, iso_pot_energy, temp_swe; };
// Exact memoisation across steps.  The snow state a step ends with (calc_snow_state at gamma_snow.h:472) is what the next
// step starts by recomputing (:411) from the same five numbers; when their bits are unchanged the result is reused.
struct GsCache {
    double k_alpha, k_scale, k_acc, k_lwc, k_tswe;  // inputs of the memoised call (NaN = empty)
    double storage, sca;                            // its outputs
    double lg_key, lg_val;                          // lgamma(alpha)
};
__device__ __forceinline__ void gs_cache_clear(GsCache& c) {
    c.k_alpha = nan_(); c.lg_key = nan_();
    c.k_scale = c.k_acc = c.k_lwc = c.k_tswe = 0.0;
    c.storage = c.sca = c.lg_val = 0.0;
}
__device__ __forceinline__ bool gs_cache_hit(GsCache& c, double alpha, double scale, double acc, double lwc, double tswe) {
    return alpha == c.k_alpha && scale == c.k_scale && acc == c.k_acc && lwc == c.k_lwc && tswe == c.k_tswe;
}
__device__ __forceinline__ void gs_cache_store(GsCache& c, double alpha, double scale, double acc, double lwc, double tswe, double storage, double sca) {
    c.k_alpha = alpha; c.k_scale = scale; c.k_acc = acc; c.k_lwc = lwc; c.k_tswe = tswe;
    c.storage = storage; c.sca = sca;
}

// The literals of the step formulas (vapour pressure, energy terms, Priestley-Taylor, unit conversions, tolerances) as a __constant__ table: sm_100a has no
// 64-bit immediate, so a double literal with a non-zero low word costs two UMOV per use (55 of the forcing-terms kernel's 420 instructions
// per step, ncu), an entry of this table one LDCU.  The same literal text as the reference, hence the same bits.
enum : int { K_VP_A = 0, K_VP_B, K_VP_C, K_VP_D, K_VP_E, K_VP_F, K_VP_G, K_VP_H, K_LW, K_LW_EXP, K_SST_A, K_SST_B, K_TURB_A, K_TURB_B, K_TURB_C,
             K_SURF_A, K_SURF_B, K_KELVIN, K_PT_CK1, K_PT_PSYCR, K_PT_BOLZ, K_PT_CK2_NEG, K_PT_CK2_POS, K_PT_CK3_NEG, K_PT_CK3_POS, K_PT_EATM_A,
             K_PT_EATM_EXP, K_PT_EATM_B, K_PT_EMIS, K_MMH_M3S, K_TOL, K_EPS_ABS, K_EPS_REL, K_Q_MIN, K_GM, K_PHYS_N };
__constant__ double kPhysC[K_PHYS_N] = {33.864, 7.38e-3, 0.8072, 1.9e-5, 1.8, 1.316e-3, 9.72e-3, 4.2e-5, 0.98 * 5.670373e-8, 6.87e-2, 1.16, 2.09, 1.7, 6.12, 6.132,
                                        0.103, 0.186, 273.15, 0.610780, 0.066, 0.0000000567, 17.84362, 17.08085, 245.425, 234.175, 1.24,
                                        0.143, 0.85, 0.98, 1 / (3600.0 * 1000.0), 1.0e-10, 1.0e-7, 1.0e-8, 0.00001, 0.001 / 86400.0};
#define SB2_K(name) kPhysC[name]
__device__ __forceinline__ double mmh_to_m3s(double mmh, double area) { return area * mmh * SB2_K(K_MMH_M3S); }  // 1 / (3600.0 * 1000.0)
__device__ __forceinline__ double m3s_to_mmh(double m3s, double area) { return m3s / (SB2_K(K_MMH_M3S) * area); }

// ---- gamma_snow ---------------------------------------------------------------------------------
// calc_q, gamma_snow.h:209-212
__device__ __forceinline__ double gs_calc_q(double a, double b, double z, double lg_a, double lg_a1) {
    const double x = z / b;
    return a * b * gamma_p<true>(a + 1.0, x, lg_a1) + z * (1.0 - gamma_p<true>(a, x, lg_a));
}

// corr_lwc = boost brent_find_minima(f, 0, z1, bits=12, 60 iterations), gamma_snow.h:214-227
__device__ __noinline__ double gs_corr_lwc(double z1, double a1, double b1, double a2, double b2) {
    const double Q1 = gs_calc_q(a1, b1, z1, sb_lgamma<true>(a1), sb_lgamma<true>(a1 + 1.0));
    const double lg_a2 = sb_lgamma<true>(a2), lg_a21 = sb_lgamma<true>(a2 + 1.0);
    // the objective (calc_q(a2, b2, z) - Q1)^2, ~10 evaluations per search: log(x) is evaluated once for both prefixes (same argument,
    // same value).  Measured and rejected (profiles/README.md): P(a2+1, x) and P(a2, x) advanced together in one pair of loops -- 7 %
    // slower in line or out of line than two calls of the single evaluation; log / exp expanded in place; the search spread over the
    // idle lanes of the warp.
    auto f = [&](double z) {
        const double x = z / b2;
        double p1 = 0.0, p0 = 0.0;  // P(a2+1, x), P(a2, x); gamma_p(): 0 unless x > 0, 1 at x = inf
        if (x == inf_()) p1 = p0 = 1.0;
        else if (x > 0.0) {
            const double lx = sb_log<true>(x);
            const double pre1 = sb_exp<true>((a2 + 1.0) * lx - x - lg_a21), pre0 = sb_exp<true>(a2 * lx - x - lg_a2);
            p1 = gamma_p_with_prefix(a2 + 1.0, x, pre1);
            p0 = gamma_p_with_prefix(a2, x, pre0);
        }
        const double d = (a2 * b2 * p1 + z * (1.0 - p0)) - Q1;
        return d * d;
    };
    const double tolerance = 0.00048828125;  // ldexp(1.0, 1 - 12)
    const double golden = (double)0.3819660f;
    double bmin = 0.0, bmax = z1;
    double x, w, v, u, delta, delta2, fu, fv, fw, fx, mid, fract1, fract2;
    x = w = v = bmax;
    fw = fv = fx = f(x);
    delta2 = delta = 0;
    int count = 60;
    do {
        mid = (bmin + bmax) / 2;
        fract1 = tolerance * fabs(x) + tolerance / 4;
        fract2 = 2 * fract1;
        if (fabs(x - mid) <= (fract2 - (bmax - bmin) / 2)) break;
        if (fabs(delta2) > fract1) {
            double r = (x - w) * (fx - fv);
            double q = (x - v) * (fx - fw);
            double p = (x - v) * q - (x - w) * r;
            q = 2 * (q - r);
            if (q > 0) p = -p;
            q = fabs(q);
            const double td = delta2;
            delta2 = delta;
            if ((fabs(p) >= fabs(q * td / 2)) || (p <= q * (bmin - x)) || (p >= q * (bmax - x))) {
                delta2 = (x >= mid) ? bmin - x : bmax - x;
                delta = golden * delta2;
            } else {
                delta = p / q;
                u = x + delta;
                if (((u - bmin) < fract2) || ((bmax - u) < fract2)) delta = (mid - x) < 0 ? -fabs(fract1) : fabs(fract1);
            }
        } else {
            delta2 = (x >= mid) ? bmin - x : bmax - x;
            delta = golden * delta2;
        }
        u = (fabs(delta) >= fract1) ? (x + delta) : (delta > 0 ? (x + fabs(fract1)) : (x - fabs(fract1)));
        fu = f(u);
        if (fu <= fx) {
            if (u >= x) bmin = x; else bmax = x;
            v = w; w = x; x = u;
            fv = fw; fw = fx; fx = fu;
        } else {
            if (u < x) bmin = u; else bmax = u;
            if ((fu <= fw) || (w == x)) {
                v = w; w = u; fv = fw; fw = fu;
            } else if ((fu <= fv) || (v == x) || (v == w)) {
                v = u; fv = fu;
            }
        }
    } while (--count);
    return x;
}

// calc_snow_state, gamma_snow.h:230-260
// `lg_key`/`lg_val` memoise lgamma(shape): the shape (alpha) changes on few steps, and equal bits in give equal bits out.
// Out of line: one copy for the three call sites of the snow step keeps that kernel inside the instruction cache (profiles/README.md, log row 15).
__device__ __noinline__ void gs_calc_snow_state(double shape, double scale, double y0, double lambda, double lwd, const InvDivisor& inv_mwf,
                                                double temp_swe, double& swe, double& sca, double& lg_key, double& lg_val) {
    const double max_water_frac = inv_mwf.d;
    double y = 0.0, y1 = 0.0;
    const double m = shape * scale;
    double lg = 0.0;
    bool have_lg = false;
    if (lambda <= 0.0) {
        swe = m;
        sca = 1.0 - y0;
    } else if (lambda / scale > 1.3 * shape + 20.0) {
        swe = sca = 0.0;
        return;
    } else {
        const double x = lambda / scale;
        if (shape != lg_key) { lg_key = shape; lg_val = sb_lgamma<true>(shape); }
        lg = lg_val;
        have_lg = true;
        const double pre = gamma_prefix<true>(shape, x, lg);
        y = (x > 0.0) ? gamma_p_with_prefix(shape, x, pre) : 0.0;
        y1 = y - pre / shape;
        swe = m * (1.0 - y1) - lambda * (1 - y);
        sca = (1.0 - y) * (1.0 - y0);
    }
    if (lwd > m) swe *= 1.0 + max_water_frac;
    else if (lwd > 0.0) {
        const double sat = div_by(lwd, inv_mwf);
        const double x = sat / scale;
        if (!have_lg) {
            if (shape != lg_key) { lg_key = shape; lg_val = sb_lgamma<true>(shape); }
            lg = lg_val;
        }
        const double pre = gamma_prefix<true>(shape, x, lg);
        const double ssa = (x == inf_()) ? 1.0 : gamma_p_with_prefix(shape, x, pre);
        const double ssa1 = ssa - pre / shape;
        const double liqwat = max_water_frac * (m * (ssa1 - y1) + sat * (1.0 - ssa) - lambda * (1.0 - y));
        swe += liqwat;
    }
    swe += temp_swe;
    swe *= 1.0 - y0;
}

// reset_snow_pack, gamma_snow.h:262-274 (alpha uses p.snow_cv, not the effective cv)
__device__ __forceinline__ void gs_reset_snow_pack(double& sca, double& lwc, double& alpha, double& sdc_melt_mean, double& acc_melt,
                                                   double& temp_swe, double storage, const PtgskParam& p) {
    if (storage > 1.0e-10) {
        sca = 1.0 - p.initial_bare_ground_fraction;
        sdc_melt_mean = storage / sca;
    } else {
        sca = sdc_melt_mean = 0.0;
    }
    alpha = 1.0 / (p.snow_cv * p.snow_cv);
    temp_swe = lwc = 0.0;
    acc_melt = -1.0;
}

// The addends of the energy balance that depend on the forcing (and parameters) only, gamma_snow.h:345-392: the long-wave term
// and the turbulent / surface-emission term.  Evaluated per step inside the fused kernel, or for a whole window by
// ptgsk_forcing_terms_kernel (no state involved); each is one addend of `effect`, so the sum keeps the reference's order.
__device__ __forceinline__ double gs_vapour_pressure(double T, double rel_hum) {
    // 33.864 * (pow(7.38e-3 * T + 0.8072, 8) - 1.9e-5 * fabs(1.8 * T + 48.0) + 1.316e-3) * rel_hum; T < 0: *= 1.0 + 9.72e-3 * T + 4.2e-5 * T * T
    double vapour_pressure = SB2_K(K_VP_A) * (sb_pow8(SB2_K(K_VP_B) * T + SB2_K(K_VP_C)) - SB2_K(K_VP_D) * fabs(SB2_K(K_VP_E) * T + 48.0) + SB2_K(K_VP_F)) * rel_hum;
    if (T < 0.0) vapour_pressure *= 1.0 + SB2_K(K_VP_G) * T + SB2_K(K_VP_H) * T * T;
    return vapour_pressure;
}
__device__ __forceinline__ void gs_energy_terms(const PtgskParam& p, double BB0, double T, double wind_speed, double rel_hum, double& lw, double& tadd) {
    const double tol = SB2_K(K_TOL);  // 1.0e-10
    // the reference's literals through kPhysC (the exponents of pow stay literals: its exact cases fold away at compile time): 273.15; 0.98 * sigma, 6.87e-2; 1.16, 2.09; 1.7, 6.12; 6.132, 0.103, 0.186
    const double T_k = T + SB2_K(K_KELVIN);
    const double turb = p.wind_scale * wind_speed + p.wind_const;
    const double vapour_pressure = gs_vapour_pressure(T, rel_hum);
    lw = SB2_K(K_LW) * sb_pow_flat<true>(vapour_pressure / T_k, 6.87e-2) * sb_pow4(T_k);
    const double sst = dmin(0.0, SB2_K(K_SST_A) * T - SB2_K(K_SST_B));
    if (sst > -tol) tadd = turb * (T + SB2_K(K_TURB_A) * (vapour_pressure - SB2_K(K_TURB_B))) - BB0;
    else tadd = turb * (T - sst + SB2_K(K_TURB_A) * (vapour_pressure - SB2_K(K_TURB_C) * sb_exp_flat<true>(SB2_K(K_SURF_A) * T - SB2_K(K_SURF_B)))) - SB2_K(K_LW) * sb_pow4(sst + SB2_K(K_KELVIN));
}

// gamma_snow::calculator::step, gamma_snow.h:291-493, given the two forcing-only addends (lw, tadd) of gs_energy_terms
// Every division by a step-invariant divisor goes through div_by (same bits as the IEEE quotient, a tenth of the instructions):
// k.inv_dt_seconds / k.inv_dt_us (the step length), the parameter-only divisors of PtgskParam, the physical constants, and inv_cv2 =
// the cell's effective snow_cv squared (p.snow_cv + forest_fraction * p.snow_cv_forest_factor + altitude * p.snow_cv_altitude_factor,
// :327; its reciprocal inv_cv2.y IS 1.0 / (snow_cv * snow_cv) of :437).
struct GsStepConst { InvDivisor inv_dt_seconds, inv_dt_us; };
__device__ __forceinline__ void gs_step_core(GsState& s, GsCache& cache, double& r_sca, double& r_storage, double& r_outflow, const PtgskParam& p, int doy,
                                             int sec_of_year, double dt_seconds, double dt_us, const GsStepConst& k, double BB0, double T, double rad,
                                             double prec_mm_h, double lw, double tadd, const double* __restrict__ f_wind_speed, const double* __restrict__ f_rel_hum,
                                             int64_t f_offset, const InvDivisor& inv_cv2) {
    const double tol = SB2_K(K_TOL);  // 1.0e-10
    const double melt_heat = 333660.0, water_heat = 4180.0, ice_heat = 2050.0;
    double sdc_melt_mean = s.sdc_melt_mean;
    double acc_melt = s.acc_melt;
    double iso_pot_energy = s.iso_pot_energy;
    const InvDivisor k_usec_per_hour = make_inv_divisor(3600000000.0), k_melt_heat = make_inv_divisor(333660.0);  // folded at compile time
    const double prec = div_by(prec_mm_h * dt_us, k_usec_per_hour);

    if (doy == p.winter_end_day_of_year) acc_melt = iso_pot_energy = 0.0;  // is_start_melt_season :95-97

    double snow, rain;
    if (T < p.tx) { snow = prec; rain = 0.0; }
    else { snow = 0.0; rain = prec; }

    if (snow < tol && sdc_melt_mean < tol && acc_melt < 0.0) {  // :313-322
        s.albedo = p.max_albedo;
        s.surface_heat = 0.0;
        s.iso_pot_energy = 0.0;
        r_sca = 0.0;
        r_storage = 0.0;
        r_outflow = prec_mm_h;
        return;
    }
    double albedo = s.albedo, lwc = s.lwc, surface_heat = s.surface_heat, alpha = s.alpha, temp_swe = s.temp_swe;
    double sca = 0.0, storage = 0.0, outflow = 0.0;

    const double min_albedo = p.min_albedo;
    const double max_albedo = p.max_albedo;
    const double albedo_range = max_albedo - min_albedo;

    if (snow > tol) albedo += div_by(snow * albedo_range, p.inv_snowfall_reset_depth);
    else {
        if (T < 0.0) albedo -= p.slow_albedo_decay_step;
        else albedo = min_albedo + p.fast_albedo_decay_step * (albedo - min_albedo);
    }
    albedo = dmax(dmin(albedo, max_albedo), min_albedo);

    double effect = rad * (1.0 - albedo);
    effect += lw;

    if (T > 0.0 && snow < tol) effect += div_by(rain * T * water_heat, k.inv_dt_seconds);
    if (T <= 0.0 && rain < tol) effect += div_by(snow * T * ice_heat, k.inv_dt_seconds);

    if (p.calculate_iso_pot_energy) {  // the only use of wind speed and relative humidity in this kernel: loaded here, under the branch
        const double wind_speed = f_wind_speed[f_offset], rel_hum = f_rel_hum[f_offset];
        const double turb = p.wind_scale * wind_speed + p.wind_const;
        const double iso_effect = effect - BB0 + turb * (T + 1.7 * (gs_vapour_pressure(T, rel_hum) - 6.12));
        iso_pot_energy += div_by(iso_effect * dt_seconds, k_melt_heat);
    }

    const double sst = dmin(0.0, 1.16 * T - 2.09);
    effect += tadd;

    double delta_sh = -surface_heat;
    surface_heat = p.surface_magnitude * ice_heat * sst * 0.5;
    delta_sh += surface_heat;

    double energy = effect * dt_seconds;
    if (delta_sh > 0.0) energy -= delta_sh;

    double potential_melt = dmax(0.0, div_by(energy, k_melt_heat));

    double sdc_scale = sdc_melt_mean / alpha;
    const double y0 = p.initial_bare_ground_fraction;
    if (gs_cache_hit(cache, alpha, sdc_scale, acc_melt, lwc, temp_swe)) {
        storage = cache.storage;
        sca = cache.sca;
    } else {
        gs_calc_snow_state(alpha, sdc_scale, y0, acc_melt, lwc, p.inv_max_water, temp_swe, storage, sca, cache.lg_key, cache.lg_val);  // cold: memo hit
        gs_cache_store(cache, alpha, sdc_scale, acc_melt, lwc, temp_swe, storage, sca);
    }
    const double start_storage_value = storage;

    if (acc_melt < 0.0) {  // :414-451
        if (snow < tol) snow = 0.0;
        else {
            const double alpha_prev = alpha;
            const double sdc_scale_prev = sdc_scale;
            const double sdc_snow = div_by(snow, p.inv_one_minus_y0);
            alpha = (sdc_melt_mean * alpha + div_by(sdc_snow, inv_cv2)) / (sdc_snow + sdc_melt_mean);
            sdc_melt_mean += sdc_snow;
            sdc_scale = sdc_melt_mean / alpha;
            if (lwc > 0.0 && sdc_snow > 0.01 * sdc_melt_mean) {
                double z1 = div_by(lwc, p.inv_max_water);
                z1 = gs_corr_lwc(z1, alpha_prev, sdc_scale_prev > 0.0 ? sdc_scale_prev : sdc_scale, alpha, sdc_scale);
                lwc = z1 * p.max_water;
                gs_calc_snow_state(alpha, sdc_scale, y0, acc_melt, lwc, p.inv_max_water, temp_swe, storage, sca, cache.lg_key, cache.lg_val);
            }
        }
        lwc += rain;
        if (sdc_melt_mean <= potential_melt) {
            storage = 0.0;
            gs_reset_snow_pack(sca, lwc, alpha, sdc_melt_mean, acc_melt, temp_swe, storage, p);
            sdc_scale = 0.0;
        } else if (potential_melt > 0.0) {
            sdc_melt_mean -= potential_melt;
            lwc += potential_melt;
            alpha = dmax(0.1, sdc_melt_mean / sdc_scale);
            if (alpha > inv_cv2.y) alpha = inv_cv2.y;  // 1.0 / (snow_cv * snow_cv)
            sdc_scale = sdc_melt_mean / alpha;
        }
    } else {  // :452-470
        temp_swe += div_by(snow, p.inv_one_minus_y0);
        if (temp_swe > 0.0) {
            const double melt = dmin(temp_swe, potential_melt);
            temp_swe -= melt;
            potential_melt -= melt;
            lwc += melt;
            if (temp_swe < tol) temp_swe = 0.0;
        }
        acc_melt += potential_melt;
        lwc += rain + potential_melt;
        // is_snow_season(t): t in [t_w_end - n_winter_days*24h, t_w_end), t_w_end = trim(t,YEAR) + winter_end_day*24h  (:89-93)
        bool in_season = true;
        if (p.calculate_iso_pot_energy) {
            const int64_t we = (int64_t)p.winter_end_day_of_year * 86400, ws = we - (int64_t)p.n_winter_days * 86400;
            in_season = (int64_t)sec_of_year >= ws && (int64_t)sec_of_year < we;
        }
        if (in_season) {
            if (storage < dmax(0.2, 2 * temp_swe) || storage < 0.2 * rain) {
                storage += snow;
                gs_reset_snow_pack(sca, lwc, alpha, sdc_melt_mean, acc_melt, temp_swe, storage, p);
                sdc_scale = sdc_melt_mean / alpha;
            }
        }
    }
    // (:472) in a cold dry spell nothing of the pack changed during the step: same five inputs, same result
    if (gs_cache_hit(cache, alpha, sdc_scale, acc_melt, lwc, temp_swe)) {
        storage = cache.storage;
        sca = cache.sca;
    } else {
        gs_calc_snow_state(alpha, sdc_scale, y0, acc_melt, lwc, p.inv_max_water, temp_swe, storage, sca, cache.lg_key, cache.lg_val);
        gs_cache_store(cache, alpha, sdc_scale, acc_melt, lwc, temp_swe, storage, sca);
    }

    outflow = prec + start_storage_value - storage;
    if (outflow < 0.0) outflow = 0.0;

    s.albedo = albedo;
    s.lwc = lwc;
    s.surface_heat = surface_heat;
    s.alpha = alpha;
    s.sdc_melt_mean = sdc_melt_mean;
    s.acc_melt = acc_melt;
    s.iso_pot_energy = iso_pot_energy;
    s.temp_swe = temp_swe;
    r_sca = sca;
    r_storage = storage;
    r_outflow = div_by(outflow * 3600000000.0, k.inv_dt_us);
}

// ---- priestley_taylor, core/priestley_taylor.h:75-103 -------------------------------------------------
__device__ __forceinline__ double pt_potential_evapotranspiration(double land_albedo, double alpha, double temperature, double global_radiation,
                                                                  double rhumidity) {
    // ck1 = 0.610780, psycr = 0.066, bolz = 0.0000000567; ck2 = 17.84362 / 17.08085 and ck3 = 245.425 / 234.175 below / above freezing (kPhysC)
    const double ck1 = SB2_K(K_PT_CK1), psycr = SB2_K(K_PT_PSYCR), bolz = SB2_K(K_PT_BOLZ);
    const bool neg = temperature < 0;
    const double ck2 = neg ? SB2_K(K_PT_CK2_NEG) : SB2_K(K_PT_CK2_POS);
    const double ck3 = neg ? SB2_K(K_PT_CK3_NEG) : SB2_K(K_PT_CK3_POS);
    const double ctt_inv = 1 / (ck3 + temperature);
    const double sat_pressure = ck1 * sb_exp_flat<true>(ck2 * temperature * ctt_inv);
    const double delta = sat_pressure * ck2 * ck3 * ctt_inv * ctt_inv;
    const double vapour_pressure = sat_pressure * rhumidity;
    const double k_temp = temperature + SB2_K(K_KELVIN);
    // 1.24 * pow(10 * vapour_pressure / k_temp, 0.143) * (0.85 + 0.5 * rhumidity);  ... (e_atm - 0.98)
    const double e_atm = SB2_K(K_PT_EATM_A) * sb_pow_flat<true>(10 * vapour_pressure / k_temp, 0.143) * (SB2_K(K_PT_EATM_B) + 0.5 * rhumidity);
    const double net_radiation = bolz * sb_pow4(k_temp) * (e_atm - SB2_K(K_PT_EMIS)) + global_radiation * (1.0 - land_albedo);
    const double epot = alpha * delta * net_radiation / (delta + psycr);
    if (epot < 0.0) return 0.0;
    return epot / (2500780 - 2361 * temperature);
}

// ---- kirchner, core/kirchner.h:186-235 --------------------------------------------------------------------
// the right-hand side d ln q / dt (kirchner.h:186-198); out of line so that the seven Runge-Kutta stages share one copy of
// the two exponentials (the step loop then stays inside the instruction cache)
__device__ __noinline__ double kirchner_rhs(double c1, double c2, double c3, double pe, double x) {
    const double g = sb_exp_inl<true>(c1 + c2 * x + c3 * x * x);  // the two exponentials interleave
    return g >= 1.e-30 ? g * (pe * sb_exp_inl<true>(-x) - 1.0) : 0.0;
}
// INL = true: the response kernel, whose whole step loop is ~1 000 instructions and stays inside the instruction cache when
// every exp/log is expanded in place (no call / argument shuffling, coefficients in uniform registers)
template <bool INL>
struct KirchnerRhs {
    double c1, c2, c3, pe;  // pe = p - e
    __device__ __forceinline__ double operator()(double x) const {
        if (INL) {
            const double g = sb_exp_inl<true>(c1 + c2 * x + c3 * x * x);
            return g >= 1.e-30 ? g * (pe * sb_exp_inl<true>(-x) - 1.0) : 0.0;
        }
        return kirchner_rhs(c1, c2, c3, pe, x);
    }
};

// runge_kutta_dopri5::calc_state: the continuous extension at theta = (t1 - t_old)/dt_old (Appendix A.2 of SURVEY.md); only reached when a
// model step took more than one sub-step, hence out of line
__device__ __noinline__ double kirchner_calc_state(double x_old, double dtl, double theta, double k1, double k3, double k4, double k5, double k6,
                                                   double k7) {
    const double c1_ = 35.0 / 384.0, c3_ = 500.0 / 1113.0, c4_ = 125.0 / 192.0, c5_ = -2187.0 / 6784.0, c6_ = 11.0 / 84.0;
    const double X1 = 5.0 * (2558722523.0 - 31403016.0 * theta) / 11282082432.0;
    const double X3 = 100.0 * (882725551.0 - 15701508.0 * theta) / 32700410799.0;
    const double X4 = 25.0 * (443332067.0 - 31403016.0 * theta) / 1880347072.0;
    const double X5 = 32805.0 * (23143187.0 - 3489224.0 * theta) / 199316789632.0;
    const double X6 = 55.0 * (29972135.0 - 7076736.0 * theta) / 822651844.0;
    const double X7 = 10.0 * (7414447.0 - 829305.0 * theta) / 29380423.0;
    const double theta_m_1 = theta - 1.0;
    const double theta_sq = theta * theta;
    const double A = theta_sq * (3.0 - 2.0 * theta);
    const double B = theta_sq * theta_m_1;
    const double C = theta_sq * theta_m_1 * theta_m_1;
    const double D = theta * theta_m_1 * theta_m_1;
    const double b1_theta = A * c1_ - C * X1 + D;
    const double b3_theta = A * c3_ + C * X3;
    const double b4_theta = A * c4_ - C * X4;
    const double b5_theta = A * c5_ + C * X5;
    const double b6_theta = A * c6_ - C * X6;
    const double b7_theta = B + C * X7;
    return 1.0 * x_old + dtl * b1_theta * k1 + dtl * b3_theta * k3 + dtl * b4_theta * k4 + dtl * b5_theta * k5 + dtl * b6_theta * k6 +
           dtl * b7_theta * k7;
}

// One model step of the log-transformed Kirchner ODE with odeint's controlled dopri5 + dense output
// (abs 1e-7, rel 1e-8): same accept/reject sequence, same step-size updates, same continuous extension.
template <bool INL = false>
__device__ __forceinline__ bool kirchner_step(double c1, double c2, double c3, double t1, double& q, double& q_avg, double p, double e) {
    const double eps_abs = SB2_K(K_EPS_ABS), eps_rel = SB2_K(K_EPS_REL);  // 1.0e-7, 1.0e-8
    if (q < SB2_K(K_Q_MIN)) q = SB2_K(K_Q_MIN);  // 0.00001
    double x = INL ? sb_log_inl<true>(q) : sb_log<true>(q);
    double t = 0.0, dt = t1;
    const KirchnerRhs<INL> rhs{c1, c2, c3, p - e};
    double dxdt = rhs(x);
    double area = 0.0, f_a = q, t_a = 0.0;

    const double b21 = 1.0 / 5.0;
    const double b31 = 3.0 / 40.0, b32 = 9.0 / 40.0;
    const double b41 = 44.0 / 45.0, b42 = -56.0 / 15.0, b43 = 32.0 / 9.0;
    const double b51 = 19372.0 / 6561.0, b52 = -25360.0 / 2187.0, b53 = 64448.0 / 6561.0, b54 = -212.0 / 729.0;
    const double b61 = 9017.0 / 3168.0, b62 = -355.0 / 33.0, b63 = 46732.0 / 5247.0, b64 = 49.0 / 176.0, b65 = -5103.0 / 18656.0;
    const double c1_ = 35.0 / 384.0, c3_ = 500.0 / 1113.0, c4_ = 125.0 / 192.0, c5_ = -2187.0 / 6784.0, c6_ = 11.0 / 84.0;
    const double dc1 = c1_ - 5179.0 / 57600.0, dc3 = c3_ - 7571.0 / 16695.0, dc4 = c4_ - 393.0 / 640.0;
    const double dc5 = c5_ - (-92097.0 / 339200.0), dc6 = c6_ - 187.0 / 2100.0, dc7 = -1.0 / 40.0;

    double x_old = x, k1 = dxdt, k3 = 0, k4 = 0, k5 = 0, k6 = 0, k7 = 0, t_old = 0.0;
    while (t < t1) {
        t_old = t;
        int fails = 0;
        double x_new, dxdt_new;
        for (;;) {
            double xt = 1.0 * x + dt * b21 * dxdt;
            const double k2 = rhs(xt);
            xt = 1.0 * x + dt * b31 * dxdt + dt * b32 * k2;
            k3 = rhs(xt);
            xt = 1.0 * x + dt * b41 * dxdt + dt * b42 * k2 + dt * b43 * k3;
            k4 = rhs(xt);
            xt = 1.0 * x + dt * b51 * dxdt + dt * b52 * k2 + dt * b53 * k3 + dt * b54 * k4;
            k5 = rhs(xt);
            xt = 1.0 * x + dt * b61 * dxdt + dt * b62 * k2 + dt * b63 * k3 + dt * b64 * k4 + dt * b65 * k5;
            k6 = rhs(xt);
            x_new = 1.0 * x + dt * c1_ * dxdt + dt * c3_ * k3 + dt * c4_ * k4 + dt * c5_ * k5 + dt * c6_ * k6;
            dxdt_new = rhs(x_new);
            const double x_err = dt * dc1 * dxdt + dt * dc3 * k3 + dt * dc4 * k4 + dt * dc5 * k5 + dt * dc6 * k6 + dt * dc7 * dxdt_new;
            const double err_num = fabs(x_err), err_den = eps_abs + eps_rel * (1.0 * fabs(x) + (1.0 * dt) * fabs(dxdt));
            // err = err_num / err_den is compared with 1 (reject) and, only when another sub-step follows, sets the next dt.
            // err_num < 0.75 err_den  =>  the rounded quotient is <= 1: accept without dividing when this sub-step reaches t1.
            if (err_num < 0.75 * err_den && !(t + dt < t1)) {
                t += dt;
                break;
            }
            const double err = err_num / err_den;
            if (err > 1.0) {
                dt *= dmax(9.0 / 10.0 * sb_pow<true>(err, -1.0 / (4 - 1)), 1.0 / 5.0);
                if (++fails >= 500) return false;
                continue;
            }
            t += dt;
            // the grown dt is only ever used by a following sub-step of this model step (initialize() resets it)
            if (err < 0.5 && t < t1) dt *= 9.0 / 10.0 * sb_pow<true>(dmax(0.00032, err), -1.0 / 5);
            break;
        }
        x_old = x; k1 = dxdt; k7 = dxdt_new;
        x = x_new; dxdt = dxdt_new;
        if (t < t1) {
            const double fq = INL ? sb_exp_inl<true>(x) : sb_exp<true>(x);
            area += 0.5 * (f_a + fq) * (t - t_a);
            f_a = fq; t_a = t;
        }
    }
    // One accepted sub-step of the whole model step (t_old = 0, t = t1; > 99.9 % of all steps): theta = 1 exactly, every b_i(theta)
    // collapses to the tableau's b_i (A = 1, B = C = D = 0, all exact) and b7(theta) = 0, i.e. calc_state(t1) is x_new bit for bit.
    if (!(t_old == 0.0 && t == t1 && fabs(k7) < inf_())) x = kirchner_calc_state(x_old, t - t_old, (t1 - t_old) / (t - t_old), k1, k3, k4, k5, k6, k7);
    q = INL ? sb_exp_inl<true>(x) : sb_exp<true>(x);
    area += 0.5 * (f_a + q) * (t1 - t_a);
    q_avg = (t1 == 1.0) ? area : area / (t1 - 0.0);  // x / 1.0 = x
    return true;
}

// Dormand-Prince tableau as odeint writes it (value_type(n)/value_type(d)); same expressions as in kirchner_step
#define SB2_DOPRI_TABLEAU { \
    1.0 / 5.0, \
    3.0 / 40.0, 9.0 / 40.0, \
    44.0 / 45.0, -56.0 / 15.0, 32.0 / 9.0, \
    19372.0 / 6561.0, -25360.0 / 2187.0, 64448.0 / 6561.0, -212.0 / 729.0, \
    9017.0 / 3168.0, -355.0 / 33.0, 46732.0 / 5247.0, 49.0 / 176.0, -5103.0 / 18656.0, \
    35.0 / 384.0, 500.0 / 1113.0, 125.0 / 192.0, -2187.0 / 6784.0, 11.0 / 84.0, \
    35.0 / 384.0 - 5179.0 / 57600.0, 500.0 / 1113.0 - 7571.0 / 16695.0, 125.0 / 192.0 - 393.0 / 640.0, \
    -2187.0 / 6784.0 - (-92097.0 / 339200.0), 11.0 / 84.0 - 187.0 / 2100.0, -1.0 / 40.0, \
    1.e-30}  /* [26]: the threshold of kirchner.h:197 */
__constant__ double kDopri[27] = SB2_DOPRI_TABLEAU;
static const double kDopri_host[27] = SB2_DOPRI_TABLEAU;
// dtb[k] = dt * tableau[k], k < 26: what the first try of every model step multiplies the slopes with (dt = t1 for all lanes then)
inline void fill_dopri_products(double dt_hours, double* dtb) {
    for (int k = 0; k < 26; ++k) dtb[k] = dt_hours * kDopri_host[k];
}

// The same step, warp-synchronous: all 32 lanes call it together and iterate until every lane has reached t1.  Each pass of the
// loop is one try_step of every lane that is still running (finished lanes recompute their last try and discard it), so the
// Runge-Kutta stages and their 14 exponentials sit in uniform control flow -- no per-lane loop, no call -- and each lane still
// follows exactly the accept / reject sequence of kirchner_step above (bit-identical; tests/test_gpu_units.py).
// DEFER: an argument outside the fast range of exp only raises `out_of_range` (the caller then repeats the whole try with DEFER = false):
// the seven stages of a try are then straight-line code without a call, and the polynomial and tableau constants can stay where they are
// between the stages instead of being fetched again after every (never taken) call site
template <bool DEFER = false>
__device__ __forceinline__ double kirchner_rhs_flat(double c1, double c2, double c3, double pe, double x, bool& out_of_range) {
    // both exponentials through one range test, so that the two polynomials interleave
    const double a = c1 + c2 * x + c3 * x * x;
    int ea, ex_;
    const double va = sb_exp_core<true>(a, ea), vx = sb_exp_core<true>(-x, ex_);
    double g = sb_scale2(va, ea);
    double ex = sb_scale2(vx, ex_);
    if (!(fabs(a) < 690.0 && fabs(x) < 690.0)) {
        if (DEFER) out_of_range = true;
        else { g = sb_exp_slow(a); ex = sb_exp_slow(-x); }
    }
    const double h = g * (pe * ex - 1.0);
    return g >= kDopri[26] ? h : 0.0;
}
__device__ __forceinline__ double kirchner_rhs_flat(double c1, double c2, double c3, double pe, double x) {
    bool unused = false;
    return kirchner_rhs_flat<false>(c1, c2, c3, pe, x, unused);
}
// One try_step of the controlled stepper from (x, dxdt) with step dt: the seven stages, the error estimate's numerator and denominator.
// UDT: dt is the same for every lane and its products with the tableau come from `dtb` (host-evaluated dt * b, the same IEEE products the
// lane would form: (dt * b21) * dxdt is how `dt * b21 * dxdt` parses) -- the first try of every model step, i.e. > 99.9 % of all tries;
// 26 fp64 multiplications less per step, and the products sit in the constant bank.
template <bool UDT, bool DEFER, class ARGS>
__device__ __forceinline__ void kirchner_try(const ARGS& ka, double dt, double c1, double c2, double c3, double pe, double x, double dxdt,
                                             double& x_new, double& dxdt_new, double& k3, double& k4, double& k5, double& k6, double& err_num,
                                             double& err_den, bool& out_of_range) {
    const double eps_abs = SB2_K(K_EPS_ABS), eps_rel = SB2_K(K_EPS_REL);  // 1.0e-7, 1.0e-8
#define SB2_DTB(k) (UDT ? ka.dtb[k] : dt * kDopri[k])
    double xt = 1.0 * x + SB2_DTB(0) * dxdt;
    const double k2 = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, xt, out_of_range);
    xt = 1.0 * x + SB2_DTB(1) * dxdt + SB2_DTB(2) * k2;
    k3 = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, xt, out_of_range);
    xt = 1.0 * x + SB2_DTB(3) * dxdt + SB2_DTB(4) * k2 + SB2_DTB(5) * k3;
    k4 = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, xt, out_of_range);
    xt = 1.0 * x + SB2_DTB(6) * dxdt + SB2_DTB(7) * k2 + SB2_DTB(8) * k3 + SB2_DTB(9) * k4;
    k5 = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, xt, out_of_range);
    xt = 1.0 * x + SB2_DTB(10) * dxdt + SB2_DTB(11) * k2 + SB2_DTB(12) * k3 + SB2_DTB(13) * k4 + SB2_DTB(14) * k5;
    k6 = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, xt, out_of_range);
    x_new = 1.0 * x + SB2_DTB(15) * dxdt + SB2_DTB(16) * k3 + SB2_DTB(17) * k4 + SB2_DTB(18) * k5 + SB2_DTB(19) * k6;
    dxdt_new = kirchner_rhs_flat<DEFER>(c1, c2, c3, pe, x_new, out_of_range);
    const double x_err = SB2_DTB(20) * dxdt + SB2_DTB(21) * k3 + SB2_DTB(22) * k4 + SB2_DTB(23) * k5 + SB2_DTB(24) * k6 + SB2_DTB(25) * dxdt_new;
#undef SB2_DTB
    err_num = fabs(x_err);
    err_den = eps_abs + eps_rel * (1.0 * fabs(x) + (1.0 * dt) * fabs(dxdt));
}
// UDT = true: t1 is the same for all lanes of the launch and ka.dtb = t1 * tableau (PtgskRunArgs::dtb / HbvRunArgs::dtb: the kernel's
// __grid_constant__ argument, read in place from the constant bank -- a pointer to it would cost an address conversion per use)
template <bool UDT, class ARGS>
__device__ __forceinline__ bool kirchner_step_warp(const ARGS& ka, double c1, double c2, double c3, double t1, double& q, double& q_avg,
                                                   double p, double e) {
    if (q < SB2_K(K_Q_MIN)) q = SB2_K(K_Q_MIN);  // 0.00001
    double x = sb_log_inl<true>(q);
    double t = 0.0, dt = t1;
    const double pe = p - e;
    double dxdt = kirchner_rhs_flat(c1, c2, c3, pe, x);
    double area = 0.0, f_a = q, t_a = 0.0;
    int fails = 0;
    bool failed = false;
    bool running = t < t1;
    // what the controller does with one try (controlled_runge_kutta::try_step + dense_output::do_step, SURVEY Appendix A.2)
    auto control = [&](double x_new, double dxdt_new, double k3, double k4, double k5, double k6, double err_num, double err_den) {
        if (!running) return;
        const double t_new = t + dt;
        if (err_num < 0.75 * err_den && !(t_new < t1)) {
            // accepted and at (or beyond) t1 without needing err itself, see kirchner_step
            if (!(t == 0.0 && t_new == t1 && fabs(dxdt_new) < inf_()))
                x = kirchner_calc_state(x, t_new - t, (t1 - t) / (t_new - t), dxdt, k3, k4, k5, k6, dxdt_new);
            else
                x = x_new;
            running = false;
            return;
        }
        const double err = err_num / err_den;
        if (err > 1.0) {
            dt *= dmax(9.0 / 10.0 * sb_pow<true>(err, -1.0 / (4 - 1)), 1.0 / 5.0);
            if (++fails >= 500) { failed = true; running = false; }
            return;
        }
        fails = 0;
        if (t_new < t1) {
            if (err < 0.5) dt *= 9.0 / 10.0 * sb_pow<true>(dmax(0.00032, err), -1.0 / 5);
            t = t_new;
            x = x_new;
            dxdt = dxdt_new;
            const double fq = sb_exp<true>(x);
            area += 0.5 * (f_a + fq) * (t - t_a);
            f_a = fq;
            t_a = t;
        } else {
            if (!(t == 0.0 && t_new == t1 && fabs(dxdt_new) < inf_()))
                x = kirchner_calc_state(x, t_new - t, (t1 - t) / (t_new - t), dxdt, k3, k4, k5, k6, dxdt_new);
            else
                x = x_new;
            running = false;
        }
    };
    double x_new, dxdt_new, k3, k4, k5, k6, err_num, err_den;
    bool out_of_range = false;
    if (UDT) {  // the first try: dt = t1 on every lane
        kirchner_try<true, true>(ka, dt, c1, c2, c3, pe, x, dxdt, x_new, dxdt_new, k3, k4, k5, k6, err_num, err_den, out_of_range);
        // an argument out of the fast range on any lane: nothing is taken from this try, and the loop below repeats it (dt = t1 still, so
        // the same products) with the full-range exp -- the same bits on the lanes that were in range
        if (!__any_sync(0xffffffffu, out_of_range)) control(x_new, dxdt_new, k3, k4, k5, k6, err_num, err_den);
    }
    while (__any_sync(0xffffffffu, running)) {
        kirchner_try<false, false>(ka, dt, c1, c2, c3, pe, x, dxdt, x_new, dxdt_new, k3, k4, k5, k6, err_num, err_den, out_of_range);
        control(x_new, dxdt_new, k3, k4, k5, k6, err_num, err_den);
    }
    q = sb_exp_flat<true>(x);
    area += 0.5 * (f_a + q) * (t1 - t_a);
    q_avg = (t1 == 1.0) ? area : area / (t1 - 0.0);  // x / 1.0 = x
    return !failed;
}

// L1 prefetch of a [step][cell] element a few steps ahead: the step kernels consume one 8-byte value per array and step, so the
// register prefetch (one step ahead) leaves the DRAM latency exposed whenever a step is short (snow-free cells, single-try steps)
__device__ __forceinline__ void prefetch_l1(const double* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#define SB2_PREFETCH_AHEAD 4   // steps; 2 and 8 measure the same, no L1 prefetch 2.5 % slower (profiles/README.md)

// ---- time slices by ticket (the five step kernels) ---------------------------------------------------------------------------
// A block steps one group of blockDim cells.  When a launch of whole-window blocks is only a few waves, the last wave leaves most of
// the machine idle for as long as a whole window takes, so the window is cut into slices of unit_steps steps: blocks take tickets
// (ticket t = cell group t % G, time slice t / G), wait until the same group's previous slice has published its state, step their
// slice and publish.  Tickets are handed out in start order, so the slice a block waits for always belongs to a block that is already
// running or done: no deadlock, and the tail shrinks to one slice.  A slice reads the state its predecessor wrote a moment ago,
// possibly on another SM: the kernels read it with __ldcg (from L2, never from a line this SM's L1 still holds from an earlier slice).
// The tickets buffer (launch_step_chunk, step_groups) holds [members] ticket counters, then [members][G] finished slices (`progress`),
// zeroed before every launch.
struct StepSlice {
    int64_t group;       // the block's cell group: cells group * blockDim.x + threadIdx.x
    int i_begin, i_end;  // its steps of the launch
    int slice;
    int* progress;       // the group's finished slices of this member; null = no time split
};
// a: the kernel's *RunArgs (n_cells, n_steps, unit_steps, tickets, progress), read in place where each field is needed; a.unit_steps == 0:
// the whole launch for cell group blockIdx.x.  The order of the locals here and of the fields of LaneSlot below is the one with which
// the kernels compile to the same SASS as when this code was written out in each of them; another order moves instructions.
template <class ARGS>
__device__ __forceinline__ StepSlice step_slice_begin(const ARGS& a, int member) {
    int64_t group = blockIdx.x;
    int* progress = nullptr;
    int slice = 0, i_begin = 0, i_end = a.n_steps;
    if (a.unit_steps > 0) {
        __shared__ int s_ticket;
        const int n_groups = int((a.n_cells + blockDim.x - 1) / blockDim.x);
        if (threadIdx.x == 0) s_ticket = atomicAdd(a.tickets + member, 1);
        __syncthreads();
        slice = s_ticket / n_groups;
        group = s_ticket - slice * n_groups;
        i_begin = slice * a.unit_steps;
        i_end = min(a.n_steps, i_begin + a.unit_steps);
        progress = a.progress + (int64_t)member * n_groups + group;
        if (threadIdx.x == 0) {
            while (*((volatile int*)progress) < slice) __nanosleep(256);
            __threadfence();
        }
        __syncthreads();
    }
    return StepSlice{group, i_begin, i_end, slice, progress};
}
// publish the slice: the block's state stores, then the counter
__device__ __forceinline__ void step_slice_publish(const StepSlice& s) {
    if (s.progress != nullptr) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) atomicExch(s.progress, s.slice + 1);
    }
}

// ---- catchment partial sums (DESIGN §3.4) ------------------------------------------------------------------------------------
// Each (warp, run of cells of one catchment) owns a slot (build_slots); per step, the lanes of a slot add their discharge and charge
// by a shuffle tree and the slot's first lane stores the sums at partial[step][slot][2].  The slots and the order of every addition
// are fixed by the cell order alone, so the sums are the same bits run to run, and in a batch member as in a single run.
// `lane` = threadIdx.x & 31 comes from the kernel: there the launch bounds limit threadIdx.x, which can fold the mask away
struct LaneSlot {
    unsigned lane;
    bool head;  // the slot's first lane: it stores the sums
    int slot;   // -1: out-of-range lane, or no partial sums
};
template <class ARGS>
__device__ __forceinline__ LaneSlot lane_slot(const ARGS& a, const double* partial, int64_t cc, bool in_range, unsigned lane) {
    LaneSlot s{lane, false, -1};
    if (partial != nullptr) {
        s.slot = in_range ? a.slot[cc] : -1;
        const int prev = __shfl_up_sync(0xffffffffu, s.slot, 1);
        s.head = in_range && (lane == 0 || prev != s.slot);
    }
    return s;
}
// every lane of the warp calls it; partial + po is the lane's slot at this step
__device__ __forceinline__ void slot_sum_store(double q, double charge, const LaneSlot& s, double* partial, int64_t po) {
    double v0 = q, v1 = charge;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const double o0 = __shfl_down_sync(0xffffffffu, v0, off);
        const double o1 = __shfl_down_sync(0xffffffffu, v1, off);
        const int os = __shfl_down_sync(0xffffffffu, s.slot, off);
        if (s.lane + off < 32 && os == s.slot) { v0 += o0; v1 += o1; }
    }
    if (s.head) {
        double* dst = partial + po;  // ((int64_t)i * n_slots + slot) * 2
        dst[0] = v0;
        dst[1] = v1;
    }
}

// ---- the phase pipeline (the production path of run_cells) ----------------------------------------------------------
// The stack of one step is a chain  forcing -> snow -> response  with no feedback from the Kirchner response into the snow
// pack, so a window of steps is run as three kernels that hand [step][cell] arrays to each other:
//   A  ptgsk_forcing_terms_kernel   stateless: Priestley-Taylor potential evapotranspiration and the two forcing-only addends of
//                                   the snow energy balance, one thread per (cell, group of steps), full occupancy
//   B  ptgsk_snow_kernel            gamma_snow over the window, eight state values in registers, data-dependent (snow / no snow,
//                                   series lengths) -- its divergence no longer stalls the ODE solver
//   C  ptgsk_response_kernel        glacier melt, actual evapotranspiration, Kirchner, discharge, catchment partial sums:
//                                   uniform control flow, few registers, many resident warps
// Same device functions, same operation order per cell as the fused kernel: results are bit-identical to it.  The extra HBM
// traffic (five scratch arrays written and read once) is paid from a memory system that the fp64-bound stack leaves >90 % idle.
#define SB2_BLOCK_A 128
#define SB2_STEPS_A 8      // steps per thread of the forcing-terms kernel
#define SB2_BLOCK_B 32
#define SB2_MINBLOCKS_B 16
#define SB2_UNIT_STEPS 128   // steps per work unit of the snow / response kernels (time split); with 4 096-step launch sets 64 / 128 / 256 measure 153.6 / 152.1 / 152.6 ms per two years
#define SB2_BLOCK_C 32
#define SB2_MINBLOCKS_C 16

// (128, 8): 63 registers, no stack, with the next step's inputs held in registers (at (128, 10) = 48 registers the prefetch spills and
// costs 1.5 %).  Without the prefetch 8, 9, 10 blocks and no bound all measure the same, (128, 1) = 94 registers costs 2.4 ms per year.
#define SB2_MINBLOCKS_A 8
template <bool UPAR>
__global__ void __launch_bounds__(SB2_BLOCK_A, SB2_MINBLOCKS_A) ptgsk_forcing_terms_kernel(const __grid_constant__ PtgskRunArgs a) {
    sb_math_stage_tables();
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_cells) return;
    if (a.active != nullptr && a.active[c] == 0) return;
    const int ens = UPAR ? 0 : blockIdx.z;  // parameter-set ensemble member (calibration); UPAR launches have none
    const PtgskParam& p = UPAR ? a.par0 : ((a.ens_params != nullptr && a.pset[c] == 0) ? a.ens_params[ens] : a.params[a.pset[c]]);
    const double pt_albedo = p.pt_albedo, pt_alpha = p.pt_alpha;
    const int64_t n = a.n_cells;
    double* __restrict__ s_pot = a.scr[SCR_POT] + (int64_t)ens * a.ens_scr_stride;
    double* __restrict__ s_lw = a.scr[SCR_LW] + (int64_t)ens * a.ens_scr_stride;
    double* __restrict__ s_tadd = a.scr[SCR_TADD] + (int64_t)ens * a.ens_scr_stride;
    const int i0 = blockIdx.y * SB2_STEPS_A;
    const int i1 = min(i0 + SB2_STEPS_A, a.n_steps);
    int64_t o = (int64_t)i0 * n + c;
    // the next step's four inputs are loaded before this step is evaluated
    double f_t = a.f[0][o], f_r = a.f[2][o], f_w = a.f[3][o], f_h = a.f[4][o];
#pragma unroll 2
    for (int i = i0; i < i1; ++i, o += n) {
        const double temp = f_t, rad = f_r, wind = f_w, rel_hum = f_h;
        if (i + 1 < i1) { const int64_t o1 = o + n; f_t = a.f[0][o1]; f_r = a.f[2][o1]; f_w = a.f[3][o1]; f_h = a.f[4][o1]; }
        double lw, tadd;
        gs_energy_terms(p, a.bb0, temp, wind, rel_hum, lw, tadd);
        s_pot[o] = pt_potential_evapotranspiration(pt_albedo, pt_alpha, temp, rad, rel_hum) * 3600.0;
        s_lw[o] = lw;
        s_tadd[o] = tadd;
    }
}

// COLLECT bits used here: 2 snow sca/swe, 4 snow_outflow, 8 state series (the eight gamma_snow fields)
// UPAR: every cell uses the region parameter set and there is no ensemble -- parameters are read from the kernel's constant bank (a.par0)
template <int COLLECT, bool UPAR>
__global__ void __launch_bounds__(SB2_BLOCK_B, SB2_MINBLOCKS_B) ptgsk_snow_kernel(const __grid_constant__ PtgskRunArgs a) {
    sb_math_stage_tables();
    const int ens = UPAR ? 0 : blockIdx.y;  // UPAR launches have no ensemble: the member offsets fold away
    // time split by ticket (1.76 waves of whole-window blocks otherwise); the memo starts empty in every slice, which costs one
    // snow-state evaluation per cell and slice
    const StepSlice sl = step_slice_begin(a, ens);
    const int i_begin = sl.i_begin, i_end = sl.i_end;
    const int64_t c = sl.group * blockDim.x + threadIdx.x;
    const bool live = c < a.n_cells && (a.active == nullptr || a.active[c] != 0);
    if (live) {
    const PtgskParam& p = UPAR ? a.par0 : ((a.ens_params != nullptr && a.pset[c] == 0) ? a.ens_params[ens] : a.params[a.pset[c]]);
    const int64_t n = a.n_cells;
    const double* __restrict__ s_lw = a.scr[SCR_LW] + (int64_t)ens * a.ens_scr_stride;
    const double* __restrict__ s_tadd = a.scr[SCR_TADD] + (int64_t)ens * a.ens_scr_stride;
    double* __restrict__ s_outflow = a.scr[SCR_OUTFLOW] + (int64_t)ens * a.ens_scr_stride;
    double* __restrict__ s_sca = a.scr[SCR_SCA] + (int64_t)ens * a.ens_scr_stride;
    const double altitude = a.z[c], cell_area_m2 = a.area[c], forest_fraction = a.forest[c];
    const double snow_storage_fraction = 1.0 - a.lake[c] - a.reservoir[c];
    // the cell's effective coefficient of variation (gamma_snow.h:327), squared, as a divisor: the same every step
    const double snow_cv = p.snow_cv + forest_fraction * p.snow_cv_forest_factor + altitude * p.snow_cv_altitude_factor;
    const InvDivisor inv_cv2 = make_inv_divisor(snow_cv * snow_cv);
    const GsStepConst gk{a.inv_dt_seconds, a.inv_dt_us};
    double* __restrict__ state = a.state + (int64_t)ens * a.ens_state_stride;
    GsState gs;
    // __ldcg: the state may have been written by the previous time slice on another SM a moment ago -- read it from L2, never from
    // a line this SM's L1 still holds from an earlier slice
    gs.albedo = __ldcg(state + 0 * n + c); gs.lwc = __ldcg(state + 1 * n + c); gs.surface_heat = __ldcg(state + 2 * n + c);
    gs.alpha = __ldcg(state + 3 * n + c); gs.sdc_melt_mean = __ldcg(state + 4 * n + c); gs.acc_melt = __ldcg(state + 5 * n + c);
    gs.iso_pot_energy = __ldcg(state + 6 * n + c); gs.temp_swe = __ldcg(state + 7 * n + c);
    GsCache cache;
    gs_cache_clear(cache);
    auto collect_state = [&](int64_t orow) {  // the state at the beginning of a step, scale_snow applied (pt_gs_k.h:213-218,367)
        a.st[1][orow] = gs.albedo;
        a.st[2][orow] = gs.lwc * snow_storage_fraction;
        a.st[3][orow] = gs.surface_heat;
        a.st[4][orow] = gs.alpha;
        a.st[5][orow] = gs.sdc_melt_mean;
        a.st[6][orow] = gs.acc_melt;
        a.st[7][orow] = gs.iso_pot_energy;
        a.st[8][orow] = gs.temp_swe * snow_storage_fraction;
    };
    // o: running element offset of (step i, cell c) in every [step][cell] array of the chunk -- bumped by n per step instead of
    // multiplied out (the 64-bit i * n + c per array access was a sixth of this kernel's instructions)
    int64_t o = (int64_t)i_begin * n + c;
    const int64_t out_shift = (a.first_step - a.out_first_step) * n;  // collected series: row of step i = local row + this (uniform)
    const int2* __restrict__ ds_row = a.day_sec_of_year + a.first_step;
    double f_t = a.f[0][o], f_p = a.f[1][o], f_r = a.f[2][o], f_lw = s_lw[o], f_ta = s_tadd[o];
    int2 f_ds = ds_row[i_begin];  // day / second of year: the step starts with a test on it, so it travels one step ahead like the forcing
    for (int i = i_begin; i < i_end; ++i, o += n) {
        const double temp = f_t, prec = f_p * p.p_corr_scale_factor, rad = f_r, lw = f_lw, tadd = f_ta;
        const int2 ds = f_ds;
        if (i + 1 < i_end) {  // the next step's inputs, one step ahead into registers
            f_ds = ds_row[i + 1];
            const int64_t o1 = o + n;
            f_t = a.f[0][o1]; f_p = a.f[1][o1]; f_r = a.f[2][o1]; f_lw = s_lw[o1]; f_ta = s_tadd[o1];
        }
        if (i + SB2_PREFETCH_AHEAD < a.n_steps) {
            const int64_t o2 = o + SB2_PREFETCH_AHEAD * n;
            prefetch_l1(a.f[0] + o2); prefetch_l1(a.f[1] + o2); prefetch_l1(a.f[2] + o2); prefetch_l1(s_lw + o2); prefetch_l1(s_tadd + o2);
        }
        const int64_t orow = o + out_shift;  // (step - a.out_first_step) * n + c
        if (COLLECT & 8) collect_state(orow);
        double sca, storage, outflow;
        gs_step_core(gs, cache, sca, storage, outflow, p, ds.x, ds.y, a.dt_seconds, a.dt_us, gk, a.bb0, temp, rad, prec, lw, tadd, a.f[3],
                     a.f[4], o, inv_cv2);
        s_outflow[o] = outflow;
        s_sca[o] = sca;
        if (COLLECT & 2) { a.resp[2][orow] = sca; a.resp[3][orow] = storage * snow_storage_fraction; }
        if (COLLECT & 4) a.resp[4][orow] = mmh_to_m3s(outflow * snow_storage_fraction, cell_area_m2);
    }
    if ((COLLECT & 8) && a.collect_end_state && i_end == a.n_steps) collect_state((a.first_step + a.n_steps - a.out_first_step) * n + c);
    state[0 * n + c] = gs.albedo; state[1 * n + c] = gs.lwc; state[2 * n + c] = gs.surface_heat; state[3 * n + c] = gs.alpha;
    state[4 * n + c] = gs.sdc_melt_mean; state[5 * n + c] = gs.acc_melt; state[6 * n + c] = gs.iso_pot_energy;
    state[7 * n + c] = gs.temp_swe;
    }  // live
    step_slice_publish(sl);
}

// COLLECT bits used here: 1 avg_discharge+charge, 4 glacier_melt/ae/pe, 8 state series (kirchner discharge)
template <int COLLECT, bool UPAR>
__global__ void __launch_bounds__(SB2_BLOCK_C, SB2_MINBLOCKS_C) ptgsk_response_kernel(const __grid_constant__ PtgskRunArgs a) {
    sb_math_stage_tables();
    const int ens = UPAR ? 0 : blockIdx.y;  // UPAR launches have no ensemble
    // time split by ticket: with ~115 registers 2 500 of the 3 125 one-warp blocks of a 100 000-cell shard are resident, so a launch of
    // whole-window blocks runs as 1.25 waves -- the second wave leaves three quarters of the machine idle for as long as the first took
    const StepSlice sl = step_slice_begin(a, ens);
    const int i_begin = sl.i_begin, i_end = sl.i_end;
    const int64_t c = sl.group * blockDim.x + threadIdx.x;
    const bool in_range = c < a.n_cells;
    const int64_t cc = in_range ? c : a.n_cells - 1;  // out-of-range lanes shadow the last cell, never store
    const bool active = in_range && (a.active == nullptr || a.active[cc] != 0);
    const unsigned lane = threadIdx.x & 31u;
    const PtgskParam& p = UPAR ? a.par0 : ((a.ens_params != nullptr && a.pset[cc] == 0) ? a.ens_params[ens] : a.params[a.pset[cc]]);
    double* __restrict__ state = a.state + (int64_t)ens * a.ens_state_stride;
    double* __restrict__ partial = a.partial != nullptr ? a.partial + (int64_t)ens * a.ens_partial_stride : nullptr;
    const double* __restrict__ s_pot = a.scr[SCR_POT] + (int64_t)ens * a.ens_scr_stride;
    const double* __restrict__ s_outflow = a.scr[SCR_OUTFLOW] + (int64_t)ens * a.ens_scr_stride;
    const double* __restrict__ s_sca = a.scr[SCR_SCA] + (int64_t)ens * a.ens_scr_stride;
    // Per-cell constants of the step (run_pt_gs_k prologue, pt_gs_k.h:347-357) live in shared memory, one column per thread: each is
    // read once or twice per step, and twelve doubles less in registers is one more resident warp per scheduler for the ODE solver.
    __shared__ double cst[14][SB2_BLOCK_C];
#define SB2_CST(k) (((volatile double*)cst[k])[threadIdx.x])
    {
        const double area = a.area[cc], gf = a.glacier[cc], lake = a.lake[cc], reservoir = a.reservoir[cc];
        const double gmd = p.gm_direct_response;
        const double drf = gf * gmd + reservoir * p.reservoir_direct_response_fraction;
        cst[0][threadIdx.x] = area;
        cst[1][threadIdx.x] = gf;
        cst[2][threadIdx.x] = gmd;
        cst[3][threadIdx.x] = 1 - gmd;
        cst[4][threadIdx.x] = 1.0 - lake - reservoir;
        cst[5][threadIdx.x] = reservoir * (1.0 - p.reservoir_direct_response_fraction) + lake;
        cst[6][threadIdx.x] = drf;
        cst[7][threadIdx.x] = 1 - drf;
        cst[8][threadIdx.x] = area * gf;
        cst[9][threadIdx.x] = p.ae_scale_factor;
        cst[10][threadIdx.x] = p.gm_dtf;
        cst[11][threadIdx.x] = p.p_corr_scale_factor;
        cst[12][threadIdx.x] = p.inv_ae_scale.y;
        cst[13][threadIdx.x] = 1.0 / (SB2_K(K_MMH_M3S) * area);  // m3s_to_mmh divides by this per-cell constant every step: div_by
    }
    const unsigned ae_e_lo = p.inv_ae_scale.e_lo;
    const unsigned mmh_e_lo = make_inv_divisor(SB2_K(K_MMH_M3S) * a.area[cc]).e_lo;
    __syncwarp();
#define cell_area_m2 SB2_CST(0)
#define glacier_fraction SB2_CST(1)
#define gm_direct SB2_CST(2)
#define gm_routed SB2_CST(3)
#define snow_storage_fraction SB2_CST(4)
#define kirchner_routed_prec SB2_CST(5)
#define direct_response_fraction SB2_CST(6)
#define kirchner_fraction SB2_CST(7)
#define glacier_area_m2 SB2_CST(8)
#define ae_scale_factor SB2_CST(9)
#define gm_dtf SB2_CST(10)
#define p_corr SB2_CST(11)
    const double c1 = p.c1, c2 = p.c2, c3 = p.c3;
    const int64_t n = a.n_cells;
    double kq = __ldcg(state + 8 * n + cc);  // L2, not L1: written by the previous time slice, possibly on another SM

    const LaneSlot ls = lane_slot(a, partial, cc, in_range, lane);
    int64_t o = (int64_t)i_begin * n + cc;  // running element offset of (step i, cell), bumped by n per step (see ptgsk_snow_kernel)
    int64_t po = ((int64_t)i_begin * a.n_slots + (ls.slot < 0 ? 0 : ls.slot)) * 2;  // likewise into partial[step][slot][2]
    const int64_t out_shift = (a.first_step - a.out_first_step) * n;
    double f_t = a.f[0][o], f_p = a.f[1][o], f_pot = s_pot[o], f_out = s_outflow[o], f_sca = s_sca[o];
    bool failed = false;
    for (int i = i_begin; i < i_end; ++i, o += n) {
        const double temp = f_t, prec = f_p * p_corr, pot = f_pot, outflow = f_out, sca = f_sca;
        if (i + 1 < i_end) {  // the next step's inputs, one step ahead into registers
            const int64_t o1 = o + n;
            f_t = a.f[0][o1]; f_p = a.f[1][o1]; f_pot = s_pot[o1]; f_out = s_outflow[o1]; f_sca = s_sca[o1];
        }
        if (i + SB2_PREFETCH_AHEAD < a.n_steps) {  // may reach into the next slice: same cells, same arrays
            const int64_t o2 = o + SB2_PREFETCH_AHEAD * n;
            prefetch_l1(a.f[0] + o2); prefetch_l1(a.f[1] + o2); prefetch_l1(s_pot + o2); prefetch_l1(s_outflow + o2);
            prefetch_l1(s_sca + o2);
        }
        const int64_t orow = o + out_shift;  // (a.first_step + i - a.out_first_step) * n + cc
        const InvDivisor inv_ae{ae_scale_factor, SB2_CST(12), ae_e_lo};
        double out_q = 0.0, out_charge = 0.0;
        {   // every lane steps (the Kirchner solver is warp-synchronous); lanes without an active cell run on benign inputs, store nothing
            if ((COLLECT & 8) && active) a.st[0][orow] = mmh_to_m3s(kq, cell_area_m2);
            // glacier_melt::step, glacier_melt.h:47-52
            const double sca_m2 = cell_area_m2 * sca;
            const double gm_melt_m3s =
                (glacier_area_m2 <= sca_m2 || temp <= 0.0) ? 0.0 : gm_dtf * temp * (glacier_area_m2 - sca_m2) * SB2_K(K_GM);  // 0.001 / 86400.0
            // actual_evapotranspiration::calculate_step, actual_evapotranspiration.h:56-62
            const double ae = pot * (1.0 - sb_exp_flat<true>(div_by(-kq * 3.0, inv_ae))) * (1.0 - dmax(sca, glacier_fraction));
            // m3s_to_mmh: the divisor is a per-cell constant, its reciprocal sits with the other per-cell constants (mostly 0 / x: no melt)
            const double gm_mmh = div_by(gm_melt_m3s, InvDivisor{SB2_K(K_MMH_M3S) * cell_area_m2, SB2_CST(13), mmh_e_lo});
            double q_avg, kq_new = active ? kq : 1.0;
            const double k_in = outflow * snow_storage_fraction + prec * kirchner_routed_prec + gm_routed * gm_mmh;
            if (!kirchner_step_warp<true>(a, c1, c2, c3, a.dt_hours, kq_new, q_avg, active ? k_in : 0.0, active ? ae : 0.0)) {
                failed = true;
                q_avg = nan("");
            }
            const double total_discharge = dmax(0.0, prec - ae) * direct_response_fraction + gm_direct * gm_mmh + q_avg * kirchner_fraction;
            const double charge_m3s =
                +mmh_to_m3s(prec, cell_area_m2) - mmh_to_m3s(ae, cell_area_m2) + gm_melt_m3s - mmh_to_m3s(total_discharge, cell_area_m2);
            if (active) {
                kq = kq_new;
                out_q = mmh_to_m3s(total_discharge, cell_area_m2);
                out_charge = charge_m3s;
                if (COLLECT & 1) { a.resp[0][orow] = out_q; a.resp[1][orow] = charge_m3s; }
                if (COLLECT & 4) {
                    a.resp[5][orow] = gm_melt_m3s;
                    a.resp[6][orow] = ae;
                    a.resp[7][orow] = pot;
                }
            }
        }
        if (partial != nullptr) {  // warp-uniform
            slot_sum_store(out_q, out_charge, ls, partial, po);
            po += 2 * a.n_slots;
        }
    }
    if (active) {
        if ((COLLECT & 8) && a.collect_end_state && i_end == a.n_steps) {
            const int64_t orow = (a.first_step + a.n_steps - a.out_first_step) * n + cc;
            a.st[0][orow] = mmh_to_m3s(kq, cell_area_m2);
        }
        state[8 * n + cc] = kq;
        if (failed) atomicOr(a.error_flag, ERR_KIRCHNER_STEP);
    }
    step_slice_publish(sl);
}
#undef cell_area_m2
#undef glacier_fraction
#undef gm_direct
#undef gm_routed
#undef snow_storage_fraction
#undef kirchner_routed_prec
#undef direct_response_fraction
#undef kirchner_fraction
#undef glacier_area_m2
#undef ae_scale_factor
#undef gm_dtf
#undef p_corr
#undef SB2_CST

// catchment sums: out[(step) * n_catch + k] = sum of the slots of catchment k, in slot order (fixed -> deterministic)
__global__ void catchment_reduce_kernel(const double* __restrict__ partial, int64_t n_slots, const int32_t* __restrict__ cat_ptr,
                                        const int32_t* __restrict__ cat_slots, int n_catch, int n_steps, double* __restrict__ out_q,
                                        double* __restrict__ out_charge, int64_t out_row0, int64_t ens_partial_stride, int64_t ens_out_stride) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n_steps * n_catch) return;
    partial += (int64_t)blockIdx.y * ens_partial_stride;  // blockIdx.y = ensemble member
    out_q += (int64_t)blockIdx.y * ens_out_stride;
    out_charge += (int64_t)blockIdx.y * ens_out_stride;
    const int i = int(idx / n_catch), k = int(idx % n_catch);
    double s0 = 0.0, s1 = 0.0;
    for (int j = cat_ptr[k]; j < cat_ptr[k + 1]; ++j) {
        const double* src = partial + ((int64_t)i * n_slots + cat_slots[j]) * 2;
        s0 += src[0];
        s1 += src[1];
    }
    out_q[(out_row0 + i) * n_catch + k] = s0;
    out_charge[(out_row0 + i) * n_catch + k] = s1;
}

}  // namespace sb2
