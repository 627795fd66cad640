// sb2_unit.cuh -- per-function evaluation kernel behind sb2_unit_eval: lets the tests compare single device functions
// (deterministic math, incomplete gamma, Brent's lwc correction, snow state, one Kirchner step) with the oracle, the way
// the reference unit-tests its methods (test/gamma_snow_test.cpp, test/kirchner_test.cpp).
#pragma once
#include "sb2_pthpsk.cuh"
#include "sb2_ptssk.cuh"

namespace sb2 {

enum { UNIT_EXP = 0, UNIT_LOG, UNIT_POW, UNIT_LGAMMA, UNIT_GAMMA_P, UNIT_CORR_LWC, UNIT_CALC_SNOW_STATE, UNIT_KIRCHNER_STEP,
       // the forms the production kernels use: branch-free exp/log/pow, the warp-synchronous Kirchner step
       UNIT_EXP_FLAT, UNIT_LOG_FLAT, UNIT_POW_FLAT, UNIT_KIRCHNER_STEP_WARP,
       // a / d through the reciprocal of a step-invariant divisor (div_by) and as the IEEE division; the Kirchner step with the host-evaluated dt * tableau
       UNIT_DIV_BY, UNIT_KIRCHNER_STEP_WARP_UDT,
       // skaugen::calculator::step: in par8 (alpha_0 d_range unit_size max_water_fraction tx cx ts cfr), state7, dt_hours, temp, prec -> state7, outflow, sca, swe, bad
       // skaugen::statistics::sca_rel_red: in u n nu_a alpha -> value, bad
       UNIT_SKAUGEN_STEP, UNIT_SCA_REL_RED,
       // hbv_physical_snow::calculator::step: in par11 (tx lw cfr wind_scale wind_const surface_magnitude max_albedo min_albedo fast / slow albedo decay
       // rate, snowfall_reset_depth), calculate_iso_pot_energy, state23 (sp sw albedo iso_pot_energy surface_heat swe sca), dt_hours, T, rad, prec, wind,
       // rel_hum -> state23, outflow, sca, storage, bad
       UNIT_HPS_STEP, UNIT_N };

__constant__ double kUnitDtb[26];  // 1.0 * tableau, uploaded by sb2_unit_eval
struct UnitDtb { struct { __device__ double operator[](int k) const { return kUnitDtb[k]; } } dtb; };

__global__ void unit_eval_kernel(int fn, int64_t n, const double* __restrict__ in, int n_in, double* __restrict__ out, int n_out) {
    sb_math_stage_tables();  // the step-kernel forms below read the tables from shared memory, the plain ones from global memory
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = i0 < n;
    const int64_t i = in_range ? i0 : n - 1;  // lanes past the end shadow the last element (warp-synchronous functions need all 32 lanes)
    const double* a = in + i * n_in;
    double ob[28];
    for (int k = 0; k < 28; ++k) ob[k] = 0.0;
    double* o = ob;
    switch (fn) {
        case UNIT_EXP: o[0] = sb_exp(a[0]); break;
        case UNIT_LOG: o[0] = sb_log(a[0]); break;
        case UNIT_POW: o[0] = sb_pow(a[0], a[1]); break;
        case UNIT_LGAMMA: o[0] = sb_lgamma(a[0]); break;
        case UNIT_GAMMA_P: o[0] = gamma_p(a[0], a[1]); break;
        case UNIT_CORR_LWC: o[0] = gs_corr_lwc(a[0], a[1], a[2], a[3], a[4]); break;
        case UNIT_CALC_SNOW_STATE: {
            double lg_key = nan_(), lg_val = 0.0;
            gs_calc_snow_state(a[0], a[1], a[2], a[3], a[4], make_inv_divisor(a[5]), a[6], o[0], o[1], lg_key, lg_val);
            break;
        }
        case UNIT_KIRCHNER_STEP: {
            double q = a[4], q_avg = 0.0;
            const bool ok = kirchner_step(a[0], a[1], a[2], a[3], q, q_avg, a[5], a[6]);
            o[0] = q; o[1] = q_avg; o[2] = ok ? 1.0 : 0.0;
            break;
        }
        case UNIT_EXP_FLAT: o[0] = sb_exp_flat<true>(a[0]); break;
        case UNIT_LOG_FLAT: o[0] = sb_log_flat<true>(a[0]); break;
        case UNIT_POW_FLAT: o[0] = sb_pow_flat<true>(a[0], a[1]); break;
        case UNIT_KIRCHNER_STEP_WARP: {
            double q = a[4], q_avg = 0.0;
            const bool ok = kirchner_step_warp<false>(UnitDtb{}, a[0], a[1], a[2], a[3], q, q_avg, a[5], a[6]);
            o[0] = q; o[1] = q_avg; o[2] = ok ? 1.0 : 0.0;
            break;
        }
        case UNIT_DIV_BY: o[0] = div_by(a[0], make_inv_divisor(a[1])); o[1] = a[0] / a[1]; break;
        case UNIT_KIRCHNER_STEP_WARP_UDT: {  // t1 = 1 hour on every lane, products from the launch's constant table (filled by the host)
            double q = a[4], q_avg = 0.0;
            const bool ok = kirchner_step_warp<true>(UnitDtb{}, a[0], a[1], a[2], 1.0, q, q_avg, a[5], a[6]);
            o[0] = q; o[1] = q_avg; o[2] = ok ? 1.0 : 0.0;
            break;
        }
        case UNIT_SKAUGEN_STEP: {
            SskParam p{};
            p.alpha_0 = a[0]; p.d_range = a[1]; p.unit_size = a[2]; p.max_water_fraction = a[3]; p.tx = a[4]; p.cx = a[5]; p.ts = a[6]; p.cfr = a[7];
            SsState s{a[8], a[9], a[10], a[11], a[12], a[13], (unsigned long long)a[14]};
            const double dt_hours = a[15];
            bool bad = false;
            ss_step(p, dt_hours, dt_hours * 3600.0 / 86400.0, make_inv_divisor(dt_hours), a[16], a[17], s, o[7], o[8], o[9], bad);
            o[0] = s.nu; o[1] = s.alpha; o[2] = s.sca; o[3] = s.swe; o[4] = s.free_water; o[5] = s.residual; o[6] = double(s.num_units);
            o[10] = bad ? 1.0 : 0.0;
            break;
        }
        case UNIT_SCA_REL_RED: {
            bool bad = false;
            o[0] = ss_sca_rel_red((unsigned long long)a[0], (unsigned long long)a[1], a[2], a[3], bad);
            o[1] = bad ? 1.0 : 0.0;
            break;
        }
        case UNIT_HPS_STEP: {
            double v[24] = {-2.439, 0.966, -0.10, 1.5, a[1], a[0], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9], a[10], a[11], 6.0, 1.0, 0.2, 1.26, 1.0, 7.0, 0.0, 1.0};
            const double dt_hours = a[35], dt_seconds = dt_hours * 3600.0;
            HpsParam p{};
            p.lw = v[4]; p.tx = v[5]; p.cfr = v[6]; p.wind_scale = v[7]; p.wind_const = v[8]; p.surface_magnitude = v[9];
            p.max_albedo = v[10]; p.min_albedo = v[11]; p.fast_albedo_decay_rate = v[12]; p.slow_albedo_decay_rate = v[13]; p.snowfall_reset_depth = v[14];
            p.calculate_iso_pot_energy = fabs(v[15]) < 0.0001 ? 0 : 1;
            for (int k = 0; k < HBV_NB; ++k) { p.I[k] = 0.25 * k; p.s[k] = 1.0; }
            const double dt_in_days = dt_seconds / 86400.0;
            p.slow_albedo_decay_step = (0.5 * (p.max_albedo - p.min_albedo) * dt_in_days / p.slow_albedo_decay_rate);
            p.fast_albedo_decay_step = sb_pow<true>(2.0, -dt_in_days / p.fast_albedo_decay_rate);
            p.inv_snowfall_reset_depth = make_inv_divisor(p.snowfall_reset_depth);
            HpsState s;
            for (int k = 0; k < HBV_NB; ++k) { s.sp[k] = a[12 + k]; s.sw[k] = a[17 + k]; s.albedo[k] = a[22 + k]; s.iso[k] = a[27 + k]; }
            s.surface_heat = a[32]; s.swe = a[33]; s.sca = a[34];
            const bool ok = hps_step(s, o[23], o[24], o[25], p, dt_seconds, dt_seconds * 1e6, 0.98 * 5.670373e-8 * sb_pow4(273.15), make_inv_divisor(dt_seconds),
                                     a[36], a[37], a[38], a[39], a[40]);
            for (int k = 0; k < HBV_NB; ++k) { o[k] = s.sp[k]; o[5 + k] = s.sw[k]; o[10 + k] = s.albedo[k]; o[15 + k] = s.iso[k]; }
            o[20] = s.surface_heat; o[21] = s.swe; o[22] = s.sca;
            o[26] = ok ? 0.0 : 1.0;
            break;
        }
        default: break;
    }
    if (in_range)
        for (int k = 0; k < n_out && k < 28; ++k) out[i * n_out + k] = ob[k];
}

}  // namespace sb2
