// sb2_pthpsk.cuh -- the pt_hps_k cell stack (Priestley-Taylor, hbv_physical_snow, actual evapotranspiration, Kirchner) on sm_100a.
//
// hbv_physical_snow keeps the five quantile bins of hbv_snow (sp, sw) and melts each of them with its own gamma_snow-type energy balance
// (albedo and iso_pot_energy per bin, one surface_heat).  One thread per cell, all 24 state values in registers, every bin loop unrolled;
// forcing prefetch as hbv_run_kernel; time slices by ticket, warp-synchronous Kirchner and segmented catchment sums from sb2_ptgsk.cuh.
//
// Follows, step for step:
//   pt_hps_k::run                              core/pt_hps_k.h:201-303
//   hbv_physical_snow::calculator::step        core/hbv_physical_snow.h:266-529 (refreeze :211-228, update_state :231-238, sca_index :240-245)
//   collectors                                 core/pt_hps_k_cell_model.h:41-230 (hps_outflow stays in mm/h, :85)
// Kept as the reference has them, because results are defined by them: sca after a snowfall is read from the redistribution FACTORS
// (p.s[i + 1], :357-362); the melt branch assigns inside its denominator, (s.sp[idx - 1] = s.sp[idx]) (:473-476); the step's updated albedo
// and surface_heat are locals that never reach the state (only a pack reset writes them).
#pragma once
#include <stdint.h>

#include "sb2_hbv.cuh"

namespace sb2 {

struct HpsParam {
    double c1, c2, c3, ae_scale_factor;
    double lw, tx, cfr, wind_scale, wind_const, surface_magnitude, max_albedo, min_albedo, fast_albedo_decay_rate, slow_albedo_decay_rate,
        snowfall_reset_depth;
    int32_t calculate_iso_pot_energy, pad_;
    double s[HBV_NB], I[HBV_NB];
    double gm_dtf, gm_direct_response, p_corr_scale_factor, pt_albedo, pt_alpha, reservoir_direct_response_fraction;
    // per-run constants the reference recomputes every step from p and dt (:300-305), evaluated once on the host
    double slow_albedo_decay_step, fast_albedo_decay_step;
    InvDivisor inv_ae_scale, inv_snowfall_reset_depth;
};
// host: parameter vector in the order of pt_hps_k::parameter::set (core/pt_hps_k.h:63-92); gm.direct_response is not part of it (default 0)
inline HpsParam make_hps_param(const double* v, int64_t dt_us) {
    HpsParam p{};
    p.c1 = v[0]; p.c2 = v[1]; p.c3 = v[2]; p.ae_scale_factor = v[3];
    p.lw = v[4]; p.tx = v[5]; p.cfr = v[6]; p.wind_scale = v[7]; p.wind_const = v[8]; p.surface_magnitude = v[9];
    p.max_albedo = v[10]; p.min_albedo = v[11]; p.fast_albedo_decay_rate = v[12]; p.slow_albedo_decay_rate = v[13]; p.snowfall_reset_depth = v[14];
    p.calculate_iso_pot_energy = std::fabs(v[15]) < 0.0001 ? 0 : 1;
    p.gm_dtf = v[16]; p.p_corr_scale_factor = v[17]; p.pt_albedo = v[18]; p.pt_alpha = v[19];
    // v[20..22] routing velocity / alpha / beta
    p.reservoir_direct_response_fraction = v[23];
    p.gm_direct_response = 0.0;  // glacier_melt::parameter default (core/glacier_melt.h)
    const double I[HBV_NB] = {0, 0.25, 0.5, 0.75, 1.0};
    double mean = 0.0;
    for (int i = 0; i < HBV_NB - 1; ++i) mean += 0.5 * (1.0 + 1.0) * (I[i + 1] - I[i]);
    for (int i = 0; i < HBV_NB; ++i) { p.I[i] = I[i]; p.s[i] = 1.0 / mean; }
    const double dt_in_days = (double(dt_us) / 1e6) / 86400.0;
    const double albedo_range = p.max_albedo - p.min_albedo;
    p.slow_albedo_decay_step = (0.5 * albedo_range * dt_in_days / p.slow_albedo_decay_rate);
    p.fast_albedo_decay_step = sb_pow(2.0, -dt_in_days / p.fast_albedo_decay_rate);
    p.inv_ae_scale = make_inv_divisor(p.ae_scale_factor);
    p.inv_snowfall_reset_depth = make_inv_divisor(p.snowfall_reset_depth);
    return p;
}

struct HpsRunArgs {
    int64_t n_cells;
    const double* __restrict__ area;
    const double* __restrict__ glacier;
    const double* __restrict__ lake;
    const double* __restrict__ reservoir;
    const int32_t* __restrict__ pset;
    const uint8_t* __restrict__ active;
    const HpsParam* __restrict__ params;
    double* __restrict__ state;  // [24][n_cells]: sp[5], sw[5], albedo[5], iso_pot_energy[5], surface_heat, swe, sca, kirchner.q
    const double* __restrict__ f[5];
    int n_steps;
    int64_t first_step;
    double dt_seconds, dt_hours, dt_us, bb0;
    double dtb[26];
    InvDivisor inv_dt_seconds;
    double* __restrict__ resp[8];
    double* __restrict__ st[4 + 4 * HBV_NB];  // kirchner_discharge, snow_sca, snow_swe, surface_heat, sp[5], sw[5], albedo[5], iso_pot_energy[5]
    int64_t out_first_step;
    int collect_end_state;
    const int32_t* __restrict__ slot;
    double* __restrict__ partial;
    int64_t n_slots;
    int* __restrict__ error_flag;
    int collect;
    int unit_steps;
    int* __restrict__ tickets;
    int* __restrict__ progress;
    // parameter-set ensemble (calibration, pthpsk_run_kernel<true>): blockIdx.y = member; member e steps its own state / partial sums
    // with the region parameter replaced by ens_params[e] (cells with a catchment override keep it, model_calibration.h:830-832);
    // tickets are [members] and progress [members][cell groups].  Last in the struct so that the fields above keep their
    // constant-bank offsets.
    const HpsParam* __restrict__ ens_params;  // null = no ensemble
    int64_t ens_state_stride, ens_partial_stride;
    int64_t ens_resp_stride;  // elements between two members' avg_discharge / charge rows (a batch that routes each member)
};

struct HpsState { double sp[HBV_NB], sw[HBV_NB], albedo[HBV_NB], iso[HBV_NB], surface_heat, swe, sca; };

// hbv_physical_snow::calculator::step (:266-529).  Returns false on "Negative outflow".
__device__ __forceinline__ bool hps_step(HpsState& s, double& r_outflow, double& r_sca, double& r_storage, const HpsParam& p, double dt_seconds, double dt_us,
                                      double BB0, const InvDivisor& inv_dt_seconds, double T, double rad, double prec_mm_h, double wind_speed,
                                      double rel_hum) {
    const double tol = 1.0e-10;
    const double water_heat = 4180.0, ice_heat = 2050.0, sigma = 5.670373e-8;
    const InvDivisor k_usec_per_hour = make_inv_divisor(3600000000.0), k_melt_heat = make_inv_divisor(333660.0);
    const double prec = div_by(prec_mm_h * dt_us, k_usec_per_hour);
    const double total_water = prec + s.swe;
    double snow, rain;
    if (T < p.tx) { snow = prec; rain = 0.0; }
    else { snow = 0.0; rain = prec; }
    s.swe += snow + s.sca * rain;
    if (s.swe < tol) {
        r_outflow = total_water;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) { s.sp[i] = s.sw[i] = 0.0; s.albedo[i] = p.max_albedo; s.iso[i] = 0.0; }
        s.swe = 0.0;
        s.sca = 0.0;
        r_sca = 0.0;
        r_storage = 0.0;
        s.surface_heat = 0.0;
        return true;
    }
    double albedo[HBV_NB];
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) albedo[i] = s.albedo[i];
    double surface_heat = s.surface_heat;
    const double min_albedo = p.min_albedo;
    const double max_albedo = p.max_albedo;
    const double albedo_range = max_albedo - min_albedo;
    const double T_k = T + 273.15;
    const double turb = p.wind_scale * wind_speed + p.wind_const;
    const double vapour_pressure = gs_vapour_pressure(T, rel_hum);  // the same expression as gamma_snow's (:306-311)
    if (snow > tol) {
        int idx = HBV_NB - 1;  // sca_index
        {
            bool found = false;
#pragma unroll
            for (int i = 0; i < HBV_NB - 1; ++i)
                if (!found && s.sca >= p.I[i] && s.sca < p.I[i + 1]) { idx = i; found = true; }
        }
        if (s.sca > 1.0e-5 && s.sca < 1.0 - 1.0e-5) {
            if (idx == 0) {
                s.sp[0] *= s.sca / (p.I[1] - p.I[0]);
                s.sw[0] *= s.sca / (p.I[1] - p.I[0]);
            } else {
#pragma unroll
                for (int i = 1; i < HBV_NB - 1; ++i)
                    if (i == idx) {
                        s.sp[i] *= (1.0 + (s.sca - p.I[i]) / (p.I[i] - p.I[i - 1])) / (1.0 + (p.I[i + 1] - p.I[i]) / (p.I[i] - p.I[i - 1]));
                        s.sw[i] *= (1.0 + (s.sca - p.I[i]) / (p.I[i] - p.I[i - 1])) / (1.0 + (p.I[i + 1] - p.I[i]) / (p.I[i] - p.I[i - 1]));
                    }
            }
        }
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {
            const double currsnow = snow * p.s[i];
            s.sp[i] += currsnow;
            albedo[i] += div_by(currsnow * albedo_range, p.inv_snowfall_reset_depth);
        }
        {   // for (i = n - 2; i > 0; --i) if (p.s[i] > 0) { sca = p.s[i + 1]; break; } else sca = p.s[1];   (sic: the factors, not the quantiles)
            bool done = false;
#pragma unroll
            for (int i = HBV_NB - 2; i > 0; --i)
                if (!done) {
                    if (p.s[i] > 0.0) { s.sca = p.s[i + 1]; done = true; }
                    else s.sca = p.s[1];
                }
        }
    } else {
        if (T < 0.0) {
#pragma unroll
            for (int i = 0; i < HBV_NB; ++i) albedo[i] -= p.slow_albedo_decay_step;
        } else {
#pragma unroll
            for (int i = 0; i < HBV_NB; ++i) albedo[i] = (min_albedo + p.fast_albedo_decay_step * (albedo[i] - min_albedo));
        }
    }
    double effect[HBV_NB];
    const double lw_term = (0.98 * sigma * sb_pow<true>(vapour_pressure / T_k, 6.87e-2) * sb_pow4(T_k));
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) {
        albedo[i] = dmax(dmin(albedo[i], max_albedo), min_albedo);
        effect[i] = rad * (1.0 - albedo[i]);
        effect[i] += lw_term;
    }
    if (T > 0.0 && snow < tol) {
        const double h = div_by(rain * T * water_heat, inv_dt_seconds);
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) effect[i] += h;
    }
    if (T <= 0.0 && rain < tol) {
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) effect[i] += div_by(snow * p.s[i] * T * ice_heat, inv_dt_seconds);
    }
    if (p.calculate_iso_pot_energy) {
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {
            const double iso_effect = (effect[i] - BB0 + turb * (T + 1.7 * (vapour_pressure - 6.12)));
            s.iso[i] += div_by(iso_effect * dt_seconds, k_melt_heat);
        }
    }
    const double sst = dmin(0.0, 1.16 * T - 2.09);
    {
        double add;
        if (sst > -tol) add = turb * (T + 1.7 * (vapour_pressure - 6.12)) - BB0;
        else add = (turb * (T - sst + 1.7 * (vapour_pressure - 6.132 * sb_exp<true>(0.103 * T - 0.186))) - 0.98 * sigma * sb_pow4(sst + 273.15));
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) effect[i] += add;
    }
    double delta_sh = -surface_heat;
    surface_heat = p.surface_magnitude * ice_heat * sst * 0.5;
    delta_sh += surface_heat;
    double potential_melt[HBV_NB];
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) {
        double energy = effect[i] * dt_seconds;
        if (delta_sh > 0.0) energy -= delta_sh;
        potential_melt[i] = div_by(energy, k_melt_heat);
    }
    const double lw = p.lw;
    int idx = HBV_NB;
    bool any_melt = false;
    {
        bool stop = false;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i)
            if (!stop && potential_melt[i] >= tol) {
                any_melt = true;
                if (s.sp[i] < potential_melt[i]) { idx = i; stop = true; }
            }
    }
    if (any_melt) {
        if (idx == 0) s.sca = 0.0;
        else if (idx == HBV_NB) s.sca = 1.0;
        else {
#pragma unroll
            for (int i = 1; i < HBV_NB; ++i)
                if (i == idx) {
                    if (s.sp[i] > 0.0) {
                        s.sp[i - 1] = s.sp[i];  // (s.sp[idx - 1] = s.sp[idx]) inside the denominator (sic)
                        s.sca = (p.I[i] - (p.I[i] - p.I[i - 1]) * (potential_melt[i] - s.sp[i]) / s.sp[i - 1]);
                    } else {
                        s.sca = (1.0 - potential_melt[i] / s.sp[i - 1]) * (s.sca - p.I[i - 1]) + p.I[i - 1];
                    }
                }
        }
    }
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) {
        if (potential_melt[i] < tol) {  // refreeze(sp, sw, rain, cfr * potential_melt, lw)
            const double potmelt = p.cfr * potential_melt[i];
            if (s.sp[i] > 0.0) {
                if (s.sw[i] + rain > -potmelt) {
                    s.sp[i] -= potmelt;
                    s.sw[i] += potmelt + rain;
                    if (s.sw[i] > s.sp[i] * lw) s.sw[i] = s.sp[i] * lw;
                } else {
                    s.sp[i] += s.sw[i] + rain;
                    s.sw[i] = 0.0;
                }
            }
        } else {  // update_state
            const double potmelt = potential_melt[i];
            if (s.sp[i] > potmelt) {
                s.sw[i] += potmelt + rain;
                s.sp[i] -= potmelt;
                s.sw[i] = dmin(s.sw[i], s.sp[i] * lw);
            } else if (s.sp[i] > 0.0) s.sp[i] = s.sw[i] = 0.0;
        }
    }
    if (s.sca < tol) s.swe = 0.0;
    else {
        const bool f_is_zero = s.sca >= 1.0 ? false : true;
        s.swe = hbv_integrate0(s.sp, p.I, s.sca, f_is_zero);
        s.swe += hbv_integrate0(s.sw, p.I, s.sca, f_is_zero);
    }
    bool ok = true;
    if (total_water < s.swe) {
        if (total_water - s.swe < -tol) ok = false;
        else s.swe = total_water;
    }
    r_outflow = total_water - s.swe;
    r_sca = s.sca;
    r_storage = s.swe;
    return ok;
}

#define SB2_HPS_MINBLOCKS 4
// ENS: a calibration batch, one grid layer per member of a.ens_params (the launcher sets the table whenever it launches this
// instantiation); without it the member is the constant 0 and every member offset folds away (the run_cells kernel)
template <bool ENS>
__global__ void __launch_bounds__(128, SB2_HPS_MINBLOCKS) pthpsk_run_kernel(const __grid_constant__ HpsRunArgs a) {
    sb_math_stage_tables();
    const int ens = ENS ? blockIdx.y : 0;
    const StepSlice sl = step_slice_begin(a, ens);
    const int i_begin = sl.i_begin, i_end = sl.i_end;
    const int64_t c = sl.group * blockDim.x + threadIdx.x;
    const bool in_range = c < a.n_cells;
    const int64_t cc = in_range ? c : a.n_cells - 1;
    const bool active = in_range && (a.active == nullptr || a.active[cc] != 0);
    const unsigned lane = threadIdx.x & 31u;
    const int64_t n = a.n_cells;
    const HpsParam& p = (ENS && a.pset[cc] == 0) ? a.ens_params[ens] : a.params[a.pset[cc]];
    const double cell_area_m2 = a.area[cc], glacier_fraction = a.glacier[cc], lake = a.lake[cc], reservoir = a.reservoir[cc];
    const double gm_direct = p.gm_direct_response;
    const double gm_routed = 1 - gm_direct;
    const double snow_storage_fraction = 1.0 - lake - reservoir;
    const double kirchner_routed_prec = reservoir * (1.0 - p.reservoir_direct_response_fraction) + lake;
    const double direct_response_fraction = glacier_fraction * gm_direct + reservoir * p.reservoir_direct_response_fraction;
    const double kirchner_fraction = 1 - direct_response_fraction;
    const double glacier_area_m2 = cell_area_m2 * glacier_fraction;

    // this member's state rows start at a.state + so, its partial sums at a.partial + ens * a.ens_partial_stride (both 0 without an ensemble)
    const int64_t so = (int64_t)ens * a.ens_state_stride;
    double* __restrict__ const resp_q = a.resp[0] + (int64_t)ens * a.ens_resp_stride;  // this member's avg_discharge / charge rows
    double* __restrict__ const resp_c = a.resp[1] + (int64_t)ens * a.ens_resp_stride;
    HpsState hs;
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) {
        hs.sp[i] = __ldcg(a.state + so + i * n + cc); hs.sw[i] = __ldcg(a.state + so + (HBV_NB + i) * n + cc);
        hs.albedo[i] = __ldcg(a.state + so + (2 * HBV_NB + i) * n + cc); hs.iso[i] = __ldcg(a.state + so + (3 * HBV_NB + i) * n + cc);
    }
    hs.surface_heat = __ldcg(a.state + so + (4 * HBV_NB) * n + cc); hs.swe = __ldcg(a.state + so + (4 * HBV_NB + 1) * n + cc);
    hs.sca = __ldcg(a.state + so + (4 * HBV_NB + 2) * n + cc);
    double kq = __ldcg(a.state + so + (4 * HBV_NB + 3) * n + cc);

    const LaneSlot ls = lane_slot(a, a.partial, cc, in_range, lane);
    auto collect_state = [&](int64_t orow) {  // state.scale_snow (pt_hps_k.h:172-176) through the state collector (pt_hps_k_cell_model.h:213-229)
        a.st[0][orow] = mmh_to_m3s(kq, cell_area_m2);
        a.st[1][orow] = hs.sca;
        a.st[2][orow] = hs.swe * snow_storage_fraction;
        a.st[3][orow] = hs.surface_heat;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {
            a.st[4 + i][orow] = hs.sp[i]; a.st[4 + HBV_NB + i][orow] = hs.sw[i];
            a.st[4 + 2 * HBV_NB + i][orow] = hs.albedo[i]; a.st[4 + 3 * HBV_NB + i][orow] = hs.iso[i];
        }
    };
    bool failed_k = false, failed_snow = false;
    int64_t o = (int64_t)i_begin * n + cc;  // running element offset of (step i, cell), bumped by n per step (see ptgsk_snow_kernel)
    const int64_t out_shift = (a.first_step - a.out_first_step) * n;
    int64_t po = (int64_t)ens * a.ens_partial_stride + ((int64_t)i_begin * a.n_slots + (ls.slot < 0 ? 0 : ls.slot)) * 2;  // likewise into partial[step][slot][2]
    double f_t = a.f[0][o], f_p = a.f[1][o], f_r = a.f[2][o], f_w = a.f[3][o], f_h = a.f[4][o];
    for (int i = i_begin; i < i_end; ++i, o += n) {
        const double temp = f_t, rad = f_r, wind = f_w, rel_hum = f_h, prec_raw = f_p;
        if (i + 1 < i_end) {
            const int64_t o1 = o + n;
            f_t = a.f[0][o1]; f_p = a.f[1][o1]; f_r = a.f[2][o1]; f_w = a.f[3][o1]; f_h = a.f[4][o1];
        }
        if (i + SB2_PREFETCH_AHEAD < a.n_steps) {
            const int64_t o2 = o + SB2_PREFETCH_AHEAD * n;
            prefetch_l1(a.f[0] + o2); prefetch_l1(a.f[1] + o2); prefetch_l1(a.f[2] + o2); prefetch_l1(a.f[3] + o2); prefetch_l1(a.f[4] + o2);
        }
        const int64_t orow = o + out_shift;  // (step - a.out_first_step) * n + cc
        double out_q = 0.0, out_charge = 0.0;
        double prec = 0.0, snow_outflow = 0.0, r_sca = 0.0, r_storage = 0.0, gm_melt_m3s = 0.0, pot = 0.0, gm_mmh = 0.0, ae = 0.0;
        if (active) {
            prec = prec_raw * p.p_corr_scale_factor;
            if (a.collect & 8) collect_state(orow);
            if (!hps_step(hs, snow_outflow, r_sca, r_storage, p, a.dt_seconds, a.dt_us, a.bb0, a.inv_dt_seconds, temp, rad, prec, wind, rel_hum)) failed_snow = true;
            const double sca_m2 = cell_area_m2 * hs.sca;
            gm_melt_m3s = (glacier_area_m2 <= sca_m2 || temp <= 0.0) ? 0.0 : p.gm_dtf * temp * (glacier_area_m2 - sca_m2) * SB2_K(K_GM);  // 0.001 / 86400.0
            pot = pt_potential_evapotranspiration(p.pt_albedo, p.pt_alpha, temp, rad, rel_hum) * 3600.0;
            gm_mmh = div_pos(gm_melt_m3s, SB2_K(K_MMH_M3S) * cell_area_m2);
            ae = pot * (1.0 - sb_exp_flat<true>(div_by(-kq * 3.0, p.inv_ae_scale))) * (1.0 - dmax(hs.sca, glacier_fraction));
        }
        double q_avg, kq_new = active ? kq : 1.0;
        const double k_in = snow_outflow * snow_storage_fraction + prec * kirchner_routed_prec + gm_routed * gm_mmh;
        if (!kirchner_step_warp<true>(a, p.c1, p.c2, p.c3, a.dt_hours, kq_new, q_avg, active ? k_in : 0.0, active ? ae : 0.0)) {
            failed_k = true;
            q_avg = nan("");
        }
        if (active) {
            kq = kq_new;
            const double total_discharge = dmax(0.0, prec - ae) * direct_response_fraction + gm_direct * gm_mmh + q_avg * kirchner_fraction;
            const double charge_m3s =
                +mmh_to_m3s(prec, cell_area_m2) - mmh_to_m3s(ae, cell_area_m2) + gm_melt_m3s - mmh_to_m3s(total_discharge, cell_area_m2);
            out_q = mmh_to_m3s(total_discharge, cell_area_m2);
            out_charge = charge_m3s;
            if (a.collect & 1) { resp_q[orow] = out_q; resp_c[orow] = charge_m3s; }
            if (a.collect & 2) { a.resp[2][orow] = r_sca; a.resp[3][orow] = r_storage * snow_storage_fraction; }
            if (a.collect & 4) {
                a.resp[4][orow] = snow_outflow * snow_storage_fraction;  // hps_outflow: mm/h, as the reference collects it
                a.resp[5][orow] = gm_melt_m3s;
                a.resp[6][orow] = ae;
                a.resp[7][orow] = pot;
            }
        }
        if (a.partial != nullptr) {
            slot_sum_store(out_q, out_charge, ls, a.partial, po);
            po += 2 * a.n_slots;
        }
    }
    if (active) {
        if ((a.collect & 8) && a.collect_end_state && i_end == a.n_steps) collect_state((a.first_step + a.n_steps - a.out_first_step) * n + cc);
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {
            a.state[so + i * n + cc] = hs.sp[i]; a.state[so + (HBV_NB + i) * n + cc] = hs.sw[i];
            a.state[so + (2 * HBV_NB + i) * n + cc] = hs.albedo[i]; a.state[so + (3 * HBV_NB + i) * n + cc] = hs.iso[i];
        }
        a.state[so + (4 * HBV_NB) * n + cc] = hs.surface_heat; a.state[so + (4 * HBV_NB + 1) * n + cc] = hs.swe;
        a.state[so + (4 * HBV_NB + 2) * n + cc] = hs.sca;
        a.state[so + (4 * HBV_NB + 3) * n + cc] = kq;
        if (failed_snow) atomicOr(a.error_flag, ERR_HBV_NEGATIVE_OUTFLOW);
        if (failed_k) atomicOr(a.error_flag, ERR_KIRCHNER_STEP);
    }
    step_slice_publish(sl);
}

}  // namespace sb2
