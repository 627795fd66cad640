// sb2_ptssk.cuh -- the pt_ss_k cell stack (Priestley-Taylor, Skaugen snow, actual evapotranspiration, Kirchner) on sm_100a.
//
// One thread per cell; the seven Skaugen state values and the Kirchner discharge stay in registers over the window, forcing and collected
// series are [time][cell]; the Kirchner step is the warp-synchronous solver of sb2_ptgsk.cuh, the time split by ticket and the catchment
// partial sums are its step_slice_begin and slot_sum_store.  The snow routine is rare, branchy work (a melt step with a partly covered cell
// searches the crossing of two gamma densities), so it sits out of line.
//
// Follows, step for step:
//   pt_ss_k::run                             core/pt_ss_k.h:195-293
//   skaugen::calculator::step                core/skaugen.h:150-339 (compute_shape_vars :341-383)
//   skaugen::statistics::sca_rel_red         core/skaugen.h:52-79 over boost 1.68 (absent from the tree): gamma_distribution pdf / cdf / mean,
//                                            tools::brent_find_minima(bits = 2), tools::bisect(eps_tolerance(10), 100 iterations) -- restated
//                                            from their published algorithms, the same restatement as oracle/sho_skaugen.hpp
//   collectors                               core/pt_ss_k_cell_model.h:41-199 (response.scale_snow / state.scale_snow, pt_ss_k.h:165-191)
#pragma once
#include <stdint.h>

#include "sb2_hbv.cuh"

namespace sb2 {

enum : int { ERR_SKAUGEN_SEARCH = 8 };  // bisect found no change of sign / gamma pdf overflow: the reference throws there

struct SskParam {
    double c1, c2, c3, ae_scale_factor;                                        // kirchner, actual_evapotranspiration
    double alpha_0, d_range, unit_size, max_water_fraction, tx, cx, ts, cfr;   // skaugen
    double p_corr_scale_factor, pt_albedo, pt_alpha;
    double gm_dtf, gm_direct_response, reservoir_direct_response_fraction;
    InvDivisor inv_ae_scale;
};
// host: parameter vector in the order of pt_ss_k::parameter::set (core/pt_ss_k.h:63-89)
inline SskParam make_ssk_param(const double* v) {
    SskParam p{};
    p.c1 = v[0]; p.c2 = v[1]; p.c3 = v[2]; p.ae_scale_factor = v[3];
    p.alpha_0 = v[4]; p.d_range = v[5]; p.unit_size = v[6]; p.max_water_fraction = v[7]; p.tx = v[8]; p.cx = v[9]; p.ts = v[10]; p.cfr = v[11];
    p.p_corr_scale_factor = v[12]; p.pt_albedo = v[13]; p.pt_alpha = v[14];
    p.gm_dtf = v[15];
    // v[16..18] routing velocity / alpha / beta: used by the routing kernels
    p.gm_direct_response = v[19]; p.reservoir_direct_response_fraction = v[20];
    p.inv_ae_scale = make_inv_divisor(p.ae_scale_factor);
    return p;
}

struct SskRunArgs {
    int64_t n_cells;
    const double* __restrict__ area;
    const double* __restrict__ glacier;
    const double* __restrict__ lake;
    const double* __restrict__ reservoir;
    const int32_t* __restrict__ pset;
    const uint8_t* __restrict__ active;
    const SskParam* __restrict__ params;
    double* __restrict__ state;  // [8][n_cells]: nu, alpha, sca, swe, free_water, residual, num_units, kirchner.q
    const double* __restrict__ f[5];
    int n_steps;
    int64_t first_step;
    double dt_seconds, dt_hours, dt_us;
    double dtb[26];              // dt_hours * Dormand-Prince tableau (kirchner_try<true>)
    InvDivisor inv_dt_hours;
    double step_in_days;
    double* __restrict__ resp[8];
    double* __restrict__ st[7];  // state series: kirchner_discharge, snow_swe, snow_sca, snow_alpha, snow_nu, snow_lwc, snow_residual
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
};

// ---- skaugen::statistics ------------------------------------------------------------------------------------------------------------
// boost gamma_distribution(shape, scale): pdf(x) = gamma_p_derivative(shape, x / scale) / scale, cdf(x) = gamma_p(shape, x / scale)
struct SsGamma {
    double shape, scale, lg;  // lg = lgamma(shape), evaluated once per distribution
    __device__ __forceinline__ double pdf(double x, bool& bad) const {
        const double z = x / scale;
        if (z == 0.0) {
            if (shape > 1.0) return 0.0;
            if (shape == 1.0) return 1.0 / scale;
            bad = true;
            return 0.0;
        }
        return sb_exp<true>(shape * sb_log<true>(z) - z - lg) / z / scale;
    }
    __device__ __forceinline__ double cdf(double x) const { return gamma_p<true>(shape, x / scale, lg); }
};
__device__ __forceinline__ int ss_sign(double v) { return v == 0.0 ? 0 : (v < 0.0 ? -1 : 1); }

// statistics::sca_rel_red (skaugen.h:52-79); `bad` is raised where the reference would throw
__device__ __noinline__ double ss_sca_rel_red(unsigned long long u, unsigned long long n, double nu_a, double alpha, bool& bad) {
    const double nu_m = (double(u) / n) * nu_a;
    const SsGamma g_m{nu_m, 1.0 / alpha, sb_lgamma<true>(nu_m)};
    const SsGamma g_a{nu_a, 1.0 / alpha, sb_lgamma<true>(nu_a)};
    const double g_a_mean = g_a.shape * g_a.scale;
    auto f = [&](double x) { return g_m.pdf(x, bad) - g_a.pdf(x, bad); };
    double lower = g_m.shape * g_m.scale;
    // upper = brent_find_minima(f, 0, g_a_mean, bits = 2).first: tolerance 2^(1-2), the iteration limit is boost's default (none)
    double upper;
    {
        const double tolerance = 0.5;
        const double golden = (double)0.3819660f;
        double bmin = 0.0, bmax = g_a_mean;
        double x, w, v, uu, delta, delta2, fu, fv, fw, fx, mid, fract1, fract2;
        x = w = v = bmax;
        fw = fv = fx = f(x);
        delta2 = delta = 0;
        long long count = 0x7fffffffLL;
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
                    uu = x + delta;
                    if (((uu - bmin) < fract2) || ((bmax - uu) < fract2)) delta = (mid - x) < 0 ? -fabs(fract1) : fabs(fract1);
                }
            } else {
                delta2 = (x >= mid) ? bmin - x : bmax - x;
                delta = golden * delta2;
            }
            uu = (fabs(delta) >= fract1) ? (x + delta) : (delta > 0 ? (x + fabs(fract1)) : (x - fabs(fract1)));
            fu = f(uu);
            if (fu <= fx) {
                if (uu >= x) bmin = x; else bmax = x;
                v = w; w = x; x = uu;
                fv = fw; fw = fx; fx = fu;
            } else {
                if (uu < x) bmin = uu; else bmax = uu;
                if ((fu <= fw) || (w == x)) {
                    v = w; w = uu; fv = fw; fw = fu;
                } else if ((fu <= fv) || (v == x) || (v == w)) {
                    v = uu; fv = fu;
                }
            }
        } while (--count);
        upper = x;
    }
    {
        int guard = 0;
        while (g_m.pdf(lower, bad) < g_a.pdf(lower, bad) && ++guard < 100000) lower *= 0.9;
    }
    // bisect(f, lower, upper, eps_tolerance<double>(10), max_iter = 100)
    double lo = lower, hi = upper;
    {
        const double eps = 0.001953125;  // max(ldexp(1.0f, 1 - 10), 4 eps)
        double fmin = f(lo), fmax = f(hi);
        if (fmin == 0.0) hi = lo;
        else if (fmax == 0.0) lo = hi;
        else if (lo >= hi || fmin * fmax >= 0.0) bad = true;
        else {
            unsigned count = 100 - 3;
            while (count && !(fabs(lo - hi) <= eps * dmin(fabs(lo), fabs(hi)))) {
                const double mid = (lo + hi) / 2;
                const double fmid = f(mid);
                if (mid == hi || mid == lo) break;
                if (fmid == 0.0) { lo = hi = mid; break; }
                else if (ss_sign(fmid) * ss_sign(fmin) < 0) { hi = mid; fmax = fmid; }
                else { lo = mid; fmin = fmid; }
                --count;
            }
        }
    }
    const double x = (lo + hi) * 0.5;
    const double m = g_m.cdf(x);
    const double a = g_a.cdf(x);
    return a + 1.0 - m;
}
__device__ __forceinline__ double ss_c(unsigned long long n, double d_range) { return sb_exp<true>(-double(n) / d_range); }  // statistics::c

// calculator::compute_shape_vars, skaugen.h:341-383
__device__ __noinline__ void ss_compute_shape_vars(double alpha_0, double d_range, double unit_size, unsigned long long nnn, unsigned long long n,
                                                   unsigned long long u, double sca, double rel_red_sca, double& alpha, double& nu) {
    const double nu_0 = alpha_0 * unit_size;
    const double dyn_var = nu / (alpha * alpha);
    const double init_var = nu_0 / (alpha_0 * alpha_0);
    double tot_var = 0.0;
    double tot_mean = 0.0;
    if (n > 0) {
        if (nnn == 0) {
            tot_var = n * init_var * (1 + (n - 1) * ss_c(n, d_range));
            tot_mean = n * nu_0 / alpha_0;
        } else {
            const double old_var_cov = (nnn + n) * init_var * (1 + ((nnn + n) - 1) * ss_c(nnn + n, d_range));
            const double new_var_cov = n * init_var * (1 + (n - 1) * ss_c(n, d_range));
            tot_var = old_var_cov * sca * sca + new_var_cov * (1.0 - sca) * (1.0 - sca);
            tot_mean = (sca * (nnn + n) + (1.0 - sca) * n) * unit_size;
        }
    }
    if (u > 0) {
        const double factor = (dyn_var / (nnn * init_var) + 1.0 + (nnn - 1) * ss_c(nnn, d_range)) / (2 * nnn);
        const double non_cond_mean = (nnn - u) * unit_size;
        tot_mean = non_cond_mean / (1.0 - rel_red_sca);
        const unsigned long long cond_u = (unsigned long long)__double2ll_rn((1.0 - rel_red_sca) * nnn - (nnn - u));
        const double auto_var = cond_u > 0 ? init_var * cond_u * (1.0 + (cond_u - 1.0) * ss_c(cond_u, d_range)) : 0.0;
        const double cross_var = cond_u > 0 ? init_var * cond_u * 2.0 * factor * cond_u : 0.0;
        tot_var = dyn_var + auto_var - cross_var;
    }
    if (fabs(tot_mean) < 1.0e-7) {
        nu = nu_0;
        alpha = alpha_0;
        return;
    }
    nu = tot_mean * tot_mean / tot_var;
    alpha = nu / (unit_size * __double2ll_rn(tot_mean / unit_size));
}

struct SsState { double nu, alpha, sca, swe, free_water, residual; unsigned long long num_units; };

// calculator::step, skaugen.h:150-339 -> outflow [mm/h], response sca and swe (over the cell); `bad` where the reference would throw
__device__ __forceinline__ void ss_step(const SskParam& p, double dt_hours, double step_in_days, const InvDivisor& inv_dt_hours, double T, double prec_mm_h,
                                     SsState& s, double& r_outflow, double& r_sca, double& r_swe, bool& bad) {
    const double snow_tol = 1.0e-10;
    const double unit_size = p.unit_size;
    const double prec = prec_mm_h * dt_hours;
    const double corr_prec = dmax(0.0, prec + s.residual);
    s.residual = dmin(0.0, prec + s.residual);
    const double snow = T < p.tx ? corr_prec : 0.0;
    const double rain = T < p.tx ? 0.0 : corr_prec;
    if (s.sca * s.swe < unit_size && snow < snow_tol) {
        r_outflow = div_by(rain + s.sca * (s.swe + s.free_water) + s.residual, inv_dt_hours);
        s.residual = 0.0;
        if (r_outflow < 0.0) {
            s.residual = r_outflow;
            r_outflow = 0.0;
        }
        s.nu = p.alpha_0 * unit_size;
        s.alpha = p.alpha_0;
        s.sca = 0.0;
        s.swe = 0.0;
        s.free_water = 0.0;
        s.num_units = 0;
        r_sca = 0.0;
        r_swe = 0.0;
        return;
    }
    const double alpha_0 = p.alpha_0;
    double swe = s.swe;
    unsigned long long nnn = s.num_units;
    double sca = s.sca;
    double nu = s.nu;
    double alpha = s.alpha;
    if (nnn > 0) nu *= nnn;
    else {
        nu = alpha_0 * p.unit_size;
        alpha = alpha_0;
    }
    double total_new_snow = snow;
    double lwc = s.free_water;
    const double total_storage = swe + lwc;
    double pot_melt = p.cx * step_in_days * (T - p.ts);
    const double refreeze = dmin(dmax(0.0, -pot_melt * p.cfr), lwc);
    total_new_snow += sca * refreeze;
    lwc -= refreeze;
    pot_melt = dmax(0.0, pot_melt);
    const double new_snow_reduction = dmin(pot_melt, total_new_snow);
    pot_melt -= new_snow_reduction;
    total_new_snow -= new_snow_reduction;
    unsigned long long n = 0;
    if (total_new_snow > unit_size) {  // 1. accumulation
        n = (unsigned long long)__double2ll_rn(total_new_snow / unit_size);
        ss_compute_shape_vars(alpha_0, p.d_range, unit_size, nnn, n, 0, sca, 0.0, alpha, nu);
        nnn = (unsigned long long)__double2ll_rn(nnn * sca) + n;
        sca = 1.0;
        swe = nnn * unit_size;
    }
    if (pot_melt > unit_size) {  // 2. melting
        unsigned long long u = (unsigned long long)__double2ll_rn(pot_melt / unit_size);
        if (nnn < u + 2) {
            nnn = 0;
            alpha = alpha_0;
            nu = alpha_0 * unit_size;
            swe = 0.0;
            lwc = 0.0;
            sca = 0.0;
        } else {
            const double rel_red_sca = ss_sca_rel_red(u, nnn, nu, alpha, bad);
            const double sca_scale_factor = 1.0 - rel_red_sca;
            sca = s.sca * sca_scale_factor;
            swe = (nnn - u) / sca_scale_factor * unit_size;
            if (swe >= nnn * unit_size) {
                u = (unsigned long long)((long long)(nnn * rel_red_sca) + 1);
                swe = (nnn - u) / sca_scale_factor * unit_size;
                if (nnn == u) sca = 0.0;
            }
            if (sca < 0.005) {
                nnn = 0;
                alpha = alpha_0;
                nu = alpha_0 * unit_size;
                swe = 0.0;
                lwc = 0.0;
                sca = 0.0;
            } else {
                ss_compute_shape_vars(alpha_0, p.d_range, unit_size, nnn, n, u, sca, rel_red_sca, alpha, nu);
                nnn = (unsigned long long)__double2ll_rn(swe / unit_size);
                swe = nnn * unit_size;
            }
        }
    }
    if (s.sca * s.swe > sca * swe) lwc += dmax(0.0, s.swe - swe);  // 3. liquid water
    lwc *= dmin(1.0, s.sca / sca);
    lwc = dmin(lwc, swe * p.max_water_fraction);
    double discharge = s.sca * total_storage + snow - sca * (swe + lwc);
    if (discharge < 0.0) {
        s.residual += discharge;
        discharge = 0.0;
    }
    if (rain > swe * p.max_water_fraction - lwc) {  // 4. rain
        discharge += sca * (rain - (swe * p.max_water_fraction - lwc)) + rain * (1.0 - sca);
        lwc = swe * p.max_water_fraction;
    } else {
        lwc += rain;
        discharge += rain * (1.0 - sca);
    }
    if (discharge >= -s.residual) {
        discharge += s.residual;
        s.residual = 0.0;
    }
    if (nnn > 0) nu /= nnn;  // 5.
    r_outflow = div_by(discharge, inv_dt_hours);
    r_swe = sca * (swe + lwc);
    r_sca = sca;
    s.nu = nu;
    s.alpha = alpha;
    s.sca = sca;
    s.swe = swe;
    s.free_water = lwc;
    s.num_units = nnn;
}

// ---- pt_ss_k::run over a chunk of steps ------------------------------------------------------------------------------------------------
// collect bits as SB2_COLLECT_*: 1 avg_discharge + charge, 2 snow sca / swe, 4 snow_outflow / glacier_melt / ae / pe, 8 state series
__global__ void __launch_bounds__(128, 4) ptssk_run_kernel(const __grid_constant__ SskRunArgs a) {
    sb_math_stage_tables();
    const StepSlice sl = step_slice_begin(a, 0);
    const int i_begin = sl.i_begin, i_end = sl.i_end;
    const int64_t c = sl.group * blockDim.x + threadIdx.x;
    const bool in_range = c < a.n_cells;
    const int64_t cc = in_range ? c : a.n_cells - 1;
    const bool active = in_range && (a.active == nullptr || a.active[cc] != 0);
    const unsigned lane = threadIdx.x & 31u;
    const int64_t n = a.n_cells;
    const SskParam& p = a.params[a.pset[cc]];
    const double cell_area_m2 = a.area[cc], glacier_fraction = a.glacier[cc], lake = a.lake[cc], reservoir = a.reservoir[cc];
    const double gm_direct = p.gm_direct_response;
    const double gm_routed = 1 - gm_direct;
    const double snow_storage_fraction = 1.0 - lake - reservoir;
    const double kirchner_routed_prec = reservoir * (1.0 - p.reservoir_direct_response_fraction) + lake;
    const double direct_response_fraction = glacier_fraction * gm_direct + reservoir * p.reservoir_direct_response_fraction;
    const double kirchner_fraction = 1 - direct_response_fraction;
    const double glacier_area_m2 = cell_area_m2 * glacier_fraction;

    SsState ss;
    ss.nu = __ldcg(a.state + 0 * n + cc); ss.alpha = __ldcg(a.state + 1 * n + cc); ss.sca = __ldcg(a.state + 2 * n + cc);
    ss.swe = __ldcg(a.state + 3 * n + cc); ss.free_water = __ldcg(a.state + 4 * n + cc); ss.residual = __ldcg(a.state + 5 * n + cc);
    ss.num_units = (unsigned long long)__ldcg(a.state + 6 * n + cc);
    double kq = __ldcg(a.state + 7 * n + cc);

    const LaneSlot ls = lane_slot(a, a.partial, cc, in_range, lane);
    auto collect_state = [&](int64_t orow) {  // state.scale_snow (pt_ss_k.h:165-171) through the state collector (pt_ss_k_cell_model.h:190-199)
        const double swe = ss.swe * snow_storage_fraction, fw = ss.free_water * snow_storage_fraction;
        a.st[0][orow] = mmh_to_m3s(kq, cell_area_m2);
        a.st[1][orow] = (fw + swe) * ss.sca;
        a.st[2][orow] = ss.sca;
        a.st[3][orow] = ss.alpha;
        a.st[4][orow] = ss.nu;
        a.st[5][orow] = fw * ss.sca;
        a.st[6][orow] = ss.residual;
    };
    bool failed_snow = false, failed_k = false;
    int64_t o = (int64_t)i_begin * n + cc;  // running element offset of (step i, cell), bumped by n per step (see ptgsk_snow_kernel)
    const int64_t out_shift = (a.first_step - a.out_first_step) * n;
    int64_t po = ((int64_t)i_begin * a.n_slots + (ls.slot < 0 ? 0 : ls.slot)) * 2;  // likewise into partial[step][slot][2]
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
        double prec = 0.0, snow_outflow = 0.0, r_sca = 0.0, r_swe = 0.0, gm_melt_m3s = 0.0, pot = 0.0, gm_mmh = 0.0, ae = 0.0;
        if (active) {
            prec = prec_raw * p.p_corr_scale_factor;
            if (a.collect & 8) collect_state(orow);
            bool bad = false;
            ss_step(p, a.dt_hours, a.step_in_days, a.inv_dt_hours, temp, prec, ss, snow_outflow, r_sca, r_swe, bad);
            failed_snow = failed_snow || bad;
            const double sca_m2 = cell_area_m2 * ss.sca;
            gm_melt_m3s = (glacier_area_m2 <= sca_m2 || temp <= 0.0) ? 0.0 : p.gm_dtf * temp * (glacier_area_m2 - sca_m2) * SB2_K(K_GM);  // 0.001 / 86400.0
            pot = pt_potential_evapotranspiration(p.pt_albedo, p.pt_alpha, temp, rad, rel_hum) * 3600.0;
            gm_mmh = div_pos(gm_melt_m3s, SB2_K(K_MMH_M3S) * cell_area_m2);
            ae = pot * (1.0 - sb_exp_flat<true>(div_by(-kq * 3.0, p.inv_ae_scale))) * (1.0 - dmax(ss.sca, glacier_fraction));
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
            if (a.collect & 1) { a.resp[0][orow] = out_q; a.resp[1][orow] = charge_m3s; }
            if (a.collect & 2) { a.resp[2][orow] = r_sca; a.resp[3][orow] = r_swe * snow_storage_fraction; }
            if (a.collect & 4) {
                a.resp[4][orow] = mmh_to_m3s(snow_outflow * snow_storage_fraction, cell_area_m2);
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
        a.state[0 * n + cc] = ss.nu; a.state[1 * n + cc] = ss.alpha; a.state[2 * n + cc] = ss.sca; a.state[3 * n + cc] = ss.swe;
        a.state[4 * n + cc] = ss.free_water; a.state[5 * n + cc] = ss.residual; a.state[6 * n + cc] = double(ss.num_units);
        a.state[7 * n + cc] = kq;
        if (failed_snow) atomicOr(a.error_flag, ERR_SKAUGEN_SEARCH);
        if (failed_k) atomicOr(a.error_flag, ERR_KIRCHNER_STEP);
    }
    step_slice_publish(sl);
}

}  // namespace sb2
