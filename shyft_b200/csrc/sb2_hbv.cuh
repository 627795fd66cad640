// sb2_hbv.cuh -- the pt_hs_k and hbv_stack cell stacks as one sm_100a kernel (template flag picks the response routine).
//
// One thread per cell; swe, sca, the five (sp, sw) snow-bin pairs and the Kirchner / soil / tank storages stay in
// registers over the window (all bin indexing is unrolled so nothing spills to local memory); forcing and collected
// series are [time][cell].
//
// Follows, step for step:
//   pt_hs_k::run                       core/pt_hs_k.h:201-283
//   hbv_stack::run_hbv_stack           core/hbv_stack.h:278-361
//   hbv_snow::calculator::step         core/hbv_snow.h:195-275 (refreeze :153-166, update_state :168-177, sca/melt index :179-193)
//   hbv_snow_common::integrate         core/hbv_snow_common.h:14-43
//   hbv_soil / hbv_tank / hbv ae       core/hbv_soil.h:59-64, core/hbv_tank.h:68-78, core/hbv_actual_evapotranspiration.h:32-38
//   collectors                         core/pt_hs_k_cell_model.h:41-208, core/hbv_stack_cell_model.h:38-215
#pragma once
#include <stdint.h>

#include "sb2_ptgsk.cuh"

namespace sb2 {

constexpr int HBV_NB = 5;  // snow bins of the default hbv_snow::parameter (core/hbv_snow.h:49-59)
enum : int { ERR_HBV_NEGATIVE_OUTFLOW = 4 };

struct HbvParam {
    double c1, c2, c3, ae_scale_factor;   // pt_hs_k: kirchner + actual_evapotranspiration
    double fc, beta, lp;                  // hbv_stack: soil + hbv actual evapotranspiration
    double uz1, kuz2, kuz1, perc, klz;    // hbv_stack: tank
    double lw, tx, cx, ts, cfr;           // hbv_snow
    double s[HBV_NB], I[HBV_NB];          // snow redistribution factors (normalised) and quantiles
    double gm_dtf, gm_direct_response;
    double p_corr_scale_factor;
    double pt_albedo, pt_alpha;
    double reservoir_direct_response_fraction;
    InvDivisor inv_lp, inv_fc, inv_ae_scale;  // parameter-only divisors with their reciprocals (div_by, sb2_math.cuh)
};

// host: parameter vectors in the order of pt_hs_k::parameter::set (core/pt_hs_k.h:66-88) / hbv_stack::parameter::set (core/hbv_stack.h:73-99)
inline HbvParam make_hbv_param(bool hbv_stack, const double* v) {
    HbvParam p{};
    if (!hbv_stack) {
        p.c1 = v[0]; p.c2 = v[1]; p.c3 = v[2]; p.ae_scale_factor = v[3];
        p.lw = v[4]; p.tx = v[5]; p.cx = v[6]; p.ts = v[7]; p.cfr = v[8];
        p.gm_dtf = v[9]; p.p_corr_scale_factor = v[10]; p.pt_albedo = v[11]; p.pt_alpha = v[12];
        p.gm_direct_response = v[16]; p.reservoir_direct_response_fraction = v[17];
    } else {
        p.fc = v[0]; p.beta = v[1]; p.lp = v[2];
        p.uz1 = v[3]; p.kuz2 = v[4]; p.kuz1 = v[5]; p.perc = v[6]; p.klz = v[7];
        p.lw = v[8]; p.tx = v[9]; p.cx = v[10]; p.ts = v[11]; p.cfr = v[12];
        p.p_corr_scale_factor = v[13]; p.pt_albedo = v[14]; p.pt_alpha = v[15]; p.gm_dtf = v[16];
        p.gm_direct_response = v[20]; p.reservoir_direct_response_fraction = v[21];
    }
    // set_std_distribution_and_quantiles + normalize_snow_distribution (core/hbv_snow.h:49-66): mean of the unit profile is 1
    const double I[HBV_NB] = {0, 0.25, 0.5, 0.75, 1.0};
    double mean = 0.0;
    for (int i = 0; i < HBV_NB - 1; ++i) mean += 0.5 * (1.0 + 1.0) * (I[i + 1] - I[i]);
    for (int i = 0; i < HBV_NB; ++i) { p.I[i] = I[i]; p.s[i] = 1.0 / mean; }
    p.inv_lp = make_inv_divisor(p.lp);
    p.inv_fc = make_inv_divisor(p.fc);
    p.inv_ae_scale = make_inv_divisor(p.ae_scale_factor);
    return p;
}

struct HbvRunArgs {
    int64_t n_cells;
    const double* __restrict__ area;
    const double* __restrict__ glacier;
    const double* __restrict__ lake;
    const double* __restrict__ reservoir;
    const int32_t* __restrict__ pset;
    const uint8_t* __restrict__ active;
    const HbvParam* __restrict__ params;
    double* __restrict__ state;  // [n_state][n_cells]
    const double* __restrict__ f[5];
    int n_steps;
    int64_t first_step;
    double dt_seconds, dt_hours, dt_us;
    double dtb[26];              // dt_hours * Dormand-Prince tableau (kirchner_try<true>, sb2_ptgsk.cuh)
    InvDivisor inv_dt_hours;     // the step length in hours as a divisor (hbv_snow's outflow, hbv_snow.h:209,272)
    double step_in_days;         // dt_seconds / 86400 (hbv_snow.h:199), host-evaluated
    HbvParam par0;               // the region parameter set by value
    double* __restrict__ resp[9];
    double* __restrict__ st[5 + 2 * HBV_NB];  // state series, ids of include/shyft_b200.h (the per-bin sp / sw series last)
    int64_t out_first_step;
    int collect_end_state;
    const int32_t* __restrict__ slot;
    double* __restrict__ partial;
    int64_t n_slots;
    int* __restrict__ error_flag;
    int collect;  // bits as SB2_COLLECT_*
    int unit_steps;              // > 0: the chunk is stepped in time slices of this many steps handed out by ticket (step_slice_begin)
    int* __restrict__ tickets;   // [1] ticket counter, zeroed per launch
    int* __restrict__ progress;  // [cell groups] finished slices per group, zeroed per launch
    // parameter-set ensemble (calibration): blockIdx.y = member; member e steps its own state / partial sums with the region
    // parameter replaced by ens_params[e] (cells with a catchment override keep it, model_calibration.h:830-832); tickets are
    // [members] and progress [members][cell groups].  Last in the struct so that the fields above keep their constant-bank offsets.
    const HbvParam* __restrict__ ens_params;  // null = no ensemble
    int64_t ens_state_stride, ens_partial_stride;
    int64_t ens_resp_stride;  // elements between two members' avg_discharge / charge rows (a batch that routes each member)
};

// hbv_snow_common::integrate(f, x, n, a = x[0], b, f_b_is_zero), core/hbv_snow_common.h:14-43
__device__ __forceinline__ double hbv_integrate0(const double (&f)[HBV_NB], const double (&x)[HBV_NB], double b, bool f_b_is_zero) {
    double area = 0.0, f_l = f[0], x_l = 0.0;
    bool done = false;
#pragma unroll
    for (int left = 0; left < HBV_NB - 1; ++left) {
        if (!done) {
            if (b >= x[left + 1]) {
                area += 0.5 * (f_l + f[left + 1]) * (x[left + 1] - x_l);
                x_l = x[left + 1];
                f_l = f[left + 1];
            } else {
                if (!f_b_is_zero) area += (f_l + 0.5 * (f[left + 1] - f_l) / (x[left + 1] - x_l) * (b - x_l)) * (b - x_l);
                else area += 0.5 * f_l * (b - x_l);
                done = true;
            }
        }
    }
    return area;
}

// hbv_snow::calculator::step, core/hbv_snow.h:195-275.  Returns false on "Negative outflow".
// dt_hours = dt_seconds / 3600 and step_in_days = dt_seconds / 86400 (:199-200) come host-evaluated; inv_dt_hours divides by dt_hours
__device__ __forceinline__ bool hbv_snow_step(double (&sp)[HBV_NB], double (&sw)[HBV_NB], double& s_swe, double& s_sca, double& outflow,
                                              const HbvParam& p, double dt_hours, double step_in_days, const InvDivisor& inv_dt_hours, double prec_mm_h,
                                              double temp) {
    double swe = s_swe, sca = s_sca;
    double I[HBV_NB];
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) I[i] = p.I[i];
    const double prec = prec_mm_h * dt_hours;
    const double total_water = prec + swe;
    double snow, rain;
    if (temp < p.tx) { snow = prec; rain = 0.0; }
    else { snow = 0.0; rain = prec; }
    swe += snow + sca * rain;
    if (swe < 0.1) {
        outflow = div_by(total_water, inv_dt_hours);
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) sp[i] = sw[i] = 0.0;
        s_swe = 0.0;
        s_sca = 0.0;
        return true;
    }
    if (snow > 0.0) {
        int idx = HBV_NB - 1;  // sca_index (:179-185)
        {
            bool found = false;
#pragma unroll
            for (int i = 0; i < HBV_NB - 1; ++i)
                if (!found && sca >= I[i] && sca < I[i + 1]) { idx = i; found = true; }
        }
        if (sca > 1.0e-5 && sca < 1.0 - 1.0e-5) {
            if (idx == 0) {
                const double k = sca / (I[1] - I[0]);
                sp[0] *= k;
                sw[0] *= k;
            } else {
#pragma unroll
                for (int i = 1; i < HBV_NB - 1; ++i)
                    if (i == idx) {
                        const double k = (1.0 + (sca - I[i]) / (I[i] - I[i - 1])) / (1.0 + (I[i + 1] - I[i]) / (I[i] - I[i - 1]));
                        sp[i] *= k;
                        sw[i] *= k;
                    }
            }
        }
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) sp[i] += snow * p.s[i];
        sca = I[1];
        {
            bool found = false;
#pragma unroll
            for (int i = HBV_NB - 2; i > 0; --i)
                if (!found && p.s[i] > 0.0) { sca = I[i + 1]; found = true; }
        }
    }
    double potmelt = p.cx * step_in_days * (temp - p.ts);
    const double lw = p.lw;
    if (potmelt < 0.0) {
        potmelt *= p.cfr;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {  // refreeze (:153-166)
            if (sp[i] > 0.0) {
                if (sw[i] + rain > -potmelt) {
                    sp[i] -= potmelt;
                    sw[i] += potmelt + rain;
                    if (sw[i] > sp[i] * lw) sw[i] = sp[i] * lw;
                } else {
                    sp[i] += sw[i] + rain;
                    sw[i] = 0.0;
                }
            }
        }
    } else {
        int idx = HBV_NB;  // melt_index (:187-193)
        {
            bool found = false;
#pragma unroll
            for (int i = 0; i < HBV_NB; ++i)
                if (!found && sp[i] < potmelt) { idx = i; found = true; }
        }
        if (idx == 0) sca = 0.0;
        else if (idx == HBV_NB) sca = 1.0;
        else {
#pragma unroll
            for (int i = 1; i < HBV_NB; ++i)
                if (i == idx) {
                    if (sp[i] > 0.0) sca = I[i] - (I[i] - I[i - 1]) * (potmelt - sp[i]) / (sp[i - 1] - sp[i]);
                    else sca = (1.0 - potmelt / sp[i - 1]) * (sca - I[i - 1]) + I[i - 1];
                }
        }
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) {  // update_state (:168-177)
            if (sp[i] > potmelt) {
                sw[i] += potmelt + rain;
                sp[i] -= potmelt;
                sw[i] = dmin(sw[i], sp[i] * lw);
            } else if (sp[i] > 0.0) sp[i] = sw[i] = 0.0;
        }
    }
    if (sca < 1.0e-6) swe = 0.0;
    else {
        const bool f_is_zero = sca >= 1.0 ? false : true;
        swe = hbv_integrate0(sp, I, sca, f_is_zero);
        swe += hbv_integrate0(sw, I, sca, f_is_zero);
    }
    bool ok = true;
    if (total_water < swe) {
        if (total_water - swe < -1.0e-6) ok = false;
        else swe = total_water;
    }
    outflow = div_by(total_water - swe, inv_dt_hours);
    s_swe = swe;
    s_sca = sca;
    return ok;
}

// launch bounds = (threads the register allocation assumes per block, blocks per SM it aims at); blocks are one warp (SB2_BLOCK), so
// (128, 4) = 128 registers -> 16 resident warps, (128, 5) = 96 registers -> 20.  Measured on 400 000 cells:
// pt_hs_k 87.8 ms at the compiler's 146 registers, 78.4 at 128, 79.4 at 96, 89.7 at 80; hbv_stack 49.1 at 122, 49.5 at 128, 46.2 at 96,
// 47.2 at 80.
#define SB2_HBV_MINBLOCKS_K 4   // pt_hs_k (Kirchner)
#define SB2_HBV_MINBLOCKS_S 5   // hbv_stack (soil + tank)
// UPAR: no catchment override in use and no ensemble -- every cell reads the region parameter set (a.par0) from the kernel's constant bank
template <bool HBV_STACK, bool UPAR>
__global__ void __launch_bounds__(128, (HBV_STACK ? SB2_HBV_MINBLOCKS_S : SB2_HBV_MINBLOCKS_K)) hbv_run_kernel(const __grid_constant__ HbvRunArgs a) {
    sb_math_stage_tables();  // exp / log tables of the shared math spec into this block's shared memory (sb2_math.cuh)
    const int ens = UPAR ? 0 : blockIdx.y;  // UPAR launches have no ensemble: the member offsets fold away
    // time split by ticket: 12 500 one-warp blocks of a 400 000-cell shard are 4-5 waves of the 2 400-3 000 resident ones, so whole-chunk
    // blocks leave a ragged last wave
    const StepSlice sl = step_slice_begin(a, ens);
    const int i_begin = sl.i_begin, i_end = sl.i_end;
    const int64_t c = sl.group * blockDim.x + threadIdx.x;
    const bool in_range = c < a.n_cells;
    const int64_t cc = in_range ? c : a.n_cells - 1;
    const bool active = in_range && (a.active == nullptr || a.active[cc] != 0);
    const unsigned lane = threadIdx.x & 31u;
    const int64_t n = a.n_cells;

    const HbvParam& p = UPAR ? a.par0 : ((a.ens_params != nullptr && a.pset[cc] == 0) ? a.ens_params[ens] : a.params[a.pset[cc]]);
    const double cell_area_m2 = a.area[cc], glacier_fraction = a.glacier[cc], lake = a.lake[cc], reservoir = a.reservoir[cc];
    const double gm_direct = p.gm_direct_response;
    const double gm_routed = 1 - gm_direct;
    const double snow_storage_fraction = 1.0 - lake - reservoir;
    const double kirchner_routed_prec = reservoir * (1.0 - p.reservoir_direct_response_fraction) + lake;
    const double direct_response_fraction = glacier_fraction * gm_direct + reservoir * p.reservoir_direct_response_fraction;
    const double land_fraction = 1 - direct_response_fraction;  // kirchner_fraction in pt_hs_k
    const double glacier_area_m2 = cell_area_m2 * glacier_fraction;

    // __ldcg: the state may have been written by the previous time slice on another SM a moment ago -- read it from L2
    // this member's state rows start at a.state + so, its partial sums at a.partial + ens * a.ens_partial_stride (both 0 without an ensemble)
    const int64_t so = (int64_t)ens * a.ens_state_stride;
    double* __restrict__ const resp_q = a.resp[0] + (int64_t)ens * a.ens_resp_stride;  // this member's avg_discharge / charge rows
    double* __restrict__ const resp_c = a.resp[1] + (int64_t)ens * a.ens_resp_stride;
    double swe = __ldcg(a.state + so + 0 * n + cc), sca = __ldcg(a.state + so + 1 * n + cc);
    double sp[HBV_NB], sw[HBV_NB];
#pragma unroll
    for (int i = 0; i < HBV_NB; ++i) { sp[i] = __ldcg(a.state + so + (2 + i) * n + cc); sw[i] = __ldcg(a.state + so + (2 + HBV_NB + i) * n + cc); }
    double x0 = __ldcg(a.state + so + (2 + 2 * HBV_NB) * n + cc);                      // kirchner.q | soil.sm
    double x1 = HBV_STACK ? __ldcg(a.state + so + (3 + 2 * HBV_NB) * n + cc) : 0.0;    // tank.uz
    double x2 = HBV_STACK ? __ldcg(a.state + so + (4 + 2 * HBV_NB) * n + cc) : 0.0;    // tank.lz

    const LaneSlot ls = lane_slot(a, a.partial, cc, in_range, lane);
    auto collect_state = [&](int64_t orow) {
        if (HBV_STACK) {  // hbv_stack_cell_model.h:196-212
            a.st[0][orow] = swe; a.st[1][orow] = sca; a.st[2][orow] = x0; a.st[3][orow] = x1; a.st[4][orow] = x2;
        } else {          // pt_hs_k_cell_model.h:193-205 on state.scale_snow (pt_hs_k.h:165-169)
            a.st[0][orow] = mmh_to_m3s(x0, cell_area_m2); a.st[1][orow] = sca; a.st[2][orow] = swe * snow_storage_fraction;
        }
        constexpr int SP0 = HBV_STACK ? 5 : 3;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) { a.st[SP0 + i][orow] = sp[i]; a.st[SP0 + HBV_NB + i][orow] = sw[i]; }  // the bins as they are (:199-202 / :209-212)
    };

    bool failed_k = false, failed_snow = false;
    // the next step's forcing is loaded one step ahead into registers and SB2_PREFETCH_AHEAD steps ahead into L1 (as the pt_gs_k kernels do):
    // the step consumes one 8-byte value per array, so without it every step waits for DRAM
    int64_t o = (int64_t)i_begin * n + cc;  // running element offset of (step i, cell), bumped by n per step (see ptgsk_snow_kernel)
    const int64_t out_shift = (a.first_step - a.out_first_step) * n;
    int64_t po = (int64_t)ens * a.ens_partial_stride + ((int64_t)i_begin * a.n_slots + (ls.slot < 0 ? 0 : ls.slot)) * 2;  // likewise into partial[step][slot][2]
    double f_t = a.f[0][o], f_p = a.f[1][o], f_r = a.f[2][o], f_h = a.f[4][o];
    for (int i = i_begin; i < i_end; ++i, o += n) {
        const double temp = f_t, rad = f_r, rel_hum = f_h, prec_raw = f_p;
        if (i + 1 < i_end) {
            const int64_t o1 = o + n;
            f_t = a.f[0][o1]; f_p = a.f[1][o1]; f_r = a.f[2][o1]; f_h = a.f[4][o1];
        }
        if (i + SB2_PREFETCH_AHEAD < a.n_steps) {
            const int64_t o2 = o + SB2_PREFETCH_AHEAD * n;
            prefetch_l1(a.f[0] + o2); prefetch_l1(a.f[1] + o2); prefetch_l1(a.f[2] + o2); prefetch_l1(a.f[4] + o2);
        }
        const int64_t orow = o + out_shift;  // (step - a.out_first_step) * n + cc
        double out_q = 0.0, out_charge = 0.0;
        // pt_hs_k: the Kirchner solver is warp-synchronous (kirchner_step_warp), so the step is split around it: every lane calls it,
        // lanes without an active cell on benign inputs
        double prec = 0.0, snow_outflow = 0.0, gm_melt_m3s = 0.0, pot = 0.0, gm_mmh = 0.0, ae = 0.0, total_discharge = 0.0, soil_outflow = 0.0;
        if (active) {
            prec = prec_raw * p.p_corr_scale_factor;
            if (a.collect & 8) collect_state(orow);
            if (!hbv_snow_step(sp, sw, swe, sca, snow_outflow, p, a.dt_hours, a.step_in_days, a.inv_dt_hours, prec, temp)) failed_snow = true;
            const double sca_m2 = cell_area_m2 * sca;
            gm_melt_m3s = (glacier_area_m2 <= sca_m2 || temp <= 0.0) ? 0.0 : p.gm_dtf * temp * (glacier_area_m2 - sca_m2) * SB2_K(K_GM);  // 0.001 / 86400.0
            pot = pt_potential_evapotranspiration(p.pt_albedo, p.pt_alpha, temp, rad, rel_hum) * 3600.0;
            gm_mmh = div_pos(gm_melt_m3s, SB2_K(K_MMH_M3S) * cell_area_m2);  // m3s_to_mmh; mostly 0 / x (no melt)
            if (HBV_STACK) {
                const double snow_fraction = dmax(sca, glacier_fraction);
                ae = (1.0 - snow_fraction) * (x0 < p.lp ? pot * div_by(x0, p.inv_lp) : pot);  // hbv_actual_evapotranspiration.h:32-38
                {  // hbv_soil::step, hbv_soil.h:59-64
                    const double t = x0 + snow_outflow;
                    const double of = snow_outflow * sb_pow<true>(div_by(t, p.inv_fc), p.beta);
                    soil_outflow = of > t ? t : of;
                    x0 = dmax(0.0, x0 + snow_outflow - soil_outflow - ae);
                }
                double tank_outflow;
                {  // hbv_tank::step, hbv_tank.h:68-78
                    const double inflow = soil_outflow + gm_routed * gm_mmh;
                    const double t = x1 + inflow;
                    const double q12 = dmax(0.0, (t - p.uz1) * p.kuz2);
                    const double q11 = dmin(t, p.uz1) * p.kuz1;
                    x1 = x1 + inflow - p.perc - (q12 + q11);
                    const double q2 = (x2 + p.perc) * p.klz;
                    x2 = x2 + p.perc - q2;
                    tank_outflow = q12 + q11 + q2;
                }
                total_discharge = dmax(0.0, prec - ae) * direct_response_fraction + gm_direct * gm_mmh + tank_outflow * land_fraction;
            } else {
                ae = pot * (1.0 - sb_exp_flat<true>(div_by(-x0 * 3.0, p.inv_ae_scale))) * (1.0 - dmax(sca, glacier_fraction));
            }
        }
        if (!HBV_STACK) {
            double q_avg, kq_new = active ? x0 : 1.0;
            const double k_in = snow_outflow * snow_storage_fraction + prec * kirchner_routed_prec + gm_routed * gm_mmh;
            if (!kirchner_step_warp<true>(a, p.c1, p.c2, p.c3, a.dt_hours, kq_new, q_avg, active ? k_in : 0.0, active ? ae : 0.0)) {
                failed_k = true;
                q_avg = nan("");
            }
            if (active) {
                x0 = kq_new;
                total_discharge = dmax(0.0, prec - ae) * direct_response_fraction + gm_direct * gm_mmh + q_avg * land_fraction;
            }
        }
        if (active) {
            const double charge_m3s =
                +mmh_to_m3s(prec, cell_area_m2) - mmh_to_m3s(ae, cell_area_m2) + gm_melt_m3s - mmh_to_m3s(total_discharge, cell_area_m2);
            out_q = mmh_to_m3s(total_discharge, cell_area_m2);
            out_charge = charge_m3s;
            if (a.collect & 1) { resp_q[orow] = out_q; resp_c[orow] = charge_m3s; }
            if (a.collect & 2) {
                // hbv_stack never assigns response.snow.snow_state (hbv_stack.h:324-357) -> its collectors record 0
                a.resp[2][orow] = HBV_STACK ? 0.0 : sca;
                a.resp[3][orow] = HBV_STACK ? 0.0 : swe * snow_storage_fraction;
            }
            if (a.collect & 4) {
                a.resp[4][orow] = HBV_STACK ? mmh_to_m3s(snow_outflow, cell_area_m2) : mmh_to_m3s(snow_outflow * snow_storage_fraction, cell_area_m2);
                a.resp[5][orow] = gm_melt_m3s;
                a.resp[6][orow] = ae;
                a.resp[7][orow] = pot;
                if (HBV_STACK) a.resp[8][orow] = soil_outflow;
            }
        }
        if (a.partial != nullptr) {
            slot_sum_store(out_q, out_charge, ls, a.partial, po);
            po += 2 * a.n_slots;
        }
    }
    if (active) {
        if ((a.collect & 8) && a.collect_end_state && i_end == a.n_steps) collect_state((a.first_step + a.n_steps - a.out_first_step) * n + cc);
        a.state[so + 0 * n + cc] = swe; a.state[so + 1 * n + cc] = sca;
#pragma unroll
        for (int i = 0; i < HBV_NB; ++i) { a.state[so + (2 + i) * n + cc] = sp[i]; a.state[so + (2 + HBV_NB + i) * n + cc] = sw[i]; }
        a.state[so + (2 + 2 * HBV_NB) * n + cc] = x0;
        if (HBV_STACK) { a.state[so + (3 + 2 * HBV_NB) * n + cc] = x1; a.state[so + (4 + 2 * HBV_NB) * n + cc] = x2; }
        if (failed_snow) atomicOr(a.error_flag, ERR_HBV_NEGATIVE_OUTFLOW);
        if (failed_k) atomicOr(a.error_flag, ERR_KIRCHNER_STEP);
    }
    step_slice_publish(sl);
}

}  // namespace sb2
