// region_model.hpp -- C++ host shim over the C ABI (include/shyft_b200.h) that keeps the member surface of the reference's
// region_model<cell_t, region_env_t> for the hot path (core/region_model.h:211-1049), so that code written against
//   model.run_interpolation(ip, ta, env); model.revert_to_initial_state(); model.run_cells(); model.catchment_discharges(cr);
// (shyft/orchestration/simulator.py:125-135 through api/boostpython/expose.h:251-290; core/model_calibration.h:830-834) keeps
// its shape.  Errors surface as std::runtime_error carrying the reference's message text.  Header-only, C++17, no CUDA headers.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <limits>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../shyft_b200.h"

namespace shyft_b200 {

using utctime = int64_t;      // microseconds since epoch (core/utctime_utilities.h:28-34)
using utctimespan = int64_t;

struct fixed_dt {  // core/time_axis.h:74-115
    utctime t = 0;
    utctimespan dt = 0;
    size_t n = 0;
    size_t size() const { return n; }
    utctime time(size_t i) const { return t + utctimespan(i) * dt; }
};

using geo_cell_data = sb2_geo_cell;                       // core/geo_cell_data.h:107-138, flattened
using interpolation_parameter = sb2_interpolation_parameter;  // core/region_model.h:65-95
inline interpolation_parameter default_interpolation_parameter() { interpolation_parameter ip; sb2_interpolation_parameter_default(&ip); return ip; }

// one variable of a_region_environment (api/api.h:137-168): geo-located series already on the model axis
struct geo_point_sources {
    std::vector<double> xyz;     // [n_sources][3]
    std::vector<double> values;  // [n_steps][n_sources]
    size_t size() const { return xyz.size() / 3; }
};
struct region_environment {
    geo_point_sources temperature, precipitation, radiation, wind_speed, rel_hum;
    const geo_point_sources& of(int var) const {
        switch (var) { case SB2_TEMPERATURE: return temperature; case SB2_PRECIPITATION: return precipitation; case SB2_RADIATION: return radiation;
                       case SB2_WIND_SPEED: return wind_speed; default: return rel_hum; }
    }
};

struct q_adjust_result {  // core/model_state_tuning.h:11-16
    double q_0 = 0.0, q_r = 0.0;
    std::string diagnostics;
};

template <int STACK>
class region_model {
    sb2_model* h_ = nullptr;
    void ck(int rc) const { if (rc != 0) throw std::runtime_error(sb2_last_error(h_)); }

  public:
    using parameter_t = std::vector<double>;            // parameter::get(i) order, size = parameter::size()
    using state_t = std::vector<double>;                // one cell's state, flat
    fixed_dt time_axis;
    interpolation_parameter ip_parameter = default_interpolation_parameter();

    // region_model(const std::vector<geo_cell_data>&, const parameter_t&)  (:283-291)
    region_model(const std::vector<geo_cell_data>& geov, const parameter_t& region_param, int device = 0) {
        if (sb2_model_create(STACK, int64_t(geov.size()), geov.data(), device, &h_) != 0) throw std::runtime_error(sb2_last_error(nullptr));
        set_region_parameter(region_param);
    }
    ~region_model() { sb2_model_destroy(h_); }
    region_model(const region_model&) = delete;
    region_model& operator=(const region_model&) = delete;
    sb2_model* handle() const { return h_; }

    size_t size() const { return size_t(sb2_size(h_)); }                                    // :860
    size_t number_of_catchments() const { return size_t(sb2_number_of_catchments(h_)); }    // :318
    std::vector<int64_t> catchment_ids() const { std::vector<int64_t> v(number_of_catchments()); ck(sb2_catchment_ids(h_, v.data())); return v; }

    void set_region_parameter(const parameter_t& p) { ck(sb2_set_region_parameter(h_, p.data(), int(p.size()))); }                       // :646-655
    parameter_t get_region_parameter() const { parameter_t p(size_t(sb2_parameter_size(h_))); ck(sb2_get_region_parameter(h_, p.data(), int(p.size()))); return p; }
    void set_catchment_parameter(int64_t cid, const parameter_t& p) { ck(sb2_set_catchment_parameter(h_, cid, p.data(), int(p.size()))); } // :668-678
    void remove_catchment_parameter(int64_t cid) { ck(sb2_remove_catchment_parameter(h_, cid)); }
    bool has_catchment_parameter(int64_t cid) const { return sb2_has_catchment_parameter(h_, cid) != 0; }
    parameter_t get_catchment_parameter(int64_t cid) const { parameter_t p(size_t(sb2_parameter_size(h_))); ck(sb2_get_catchment_parameter(h_, cid, p.data(), int(p.size()))); return p; }
    void set_catchment_calculation_filter(const std::vector<int64_t>& cids) { ck(sb2_set_catchment_calculation_filter(h_, cids.data(), int(cids.size()))); }  // :715-729

    // states: vector<state_t> flattened [cell][state_size]
    void set_states(const std::vector<double>& states) {                                                                                       // :802-809
        const size_t ss = size_t(sb2_state_size(h_));
        if (states.size() % ss != 0) throw std::runtime_error("set_states: the flattened state vector is not a whole number of cell states");
        ck(sb2_set_states(h_, states.data(), int64_t(states.size() / ss)));  // a wrong cell count is the reference's "Length of the state vector ..." error
    }
    void get_states(std::vector<double>& states) const { states.resize(size() * size_t(sb2_state_size(h_))); ck(sb2_get_states(h_, states.data(), int64_t(size()))); }
    void revert_to_initial_state() { ck(sb2_revert_to_initial_state(h_)); }                                                                   // :814-818
    void adjust_q(double q_scale, const std::vector<int64_t>& cids) { ck(sb2_adjust_q(h_, q_scale, cids.data(), int(cids.size()))); }          // :831-837
    void set_collector_mode(int bits) { ck(sb2_set_collector_mode(h_, bits)); }
    // state_io_handler (api/api_state.h:93-142): ids and flattened states of the cells of `cids`; apply returns the unmatched positions
    void extract_state(const std::vector<int64_t>& cids, std::vector<sb2_cell_state_id>& ids, std::vector<double>& states) const {
        ids.resize(size());
        states.resize(size() * size_t(sb2_state_size(h_)));
        int64_t n = 0;
        ck(sb2_extract_state(h_, cids.data(), int(cids.size()), ids.data(), states.data(), &n));
        ids.resize(size_t(n));
        states.resize(size_t(n) * size_t(sb2_state_size(h_)));
    }
    std::vector<int64_t> apply_state(const std::vector<sb2_cell_state_id>& ids, const std::vector<double>& states, const std::vector<int64_t>& cids) {
        std::vector<int64_t> missing(ids.size() + 1);
        int64_t n = 0;
        if (states.size() != ids.size() * size_t(sb2_state_size(h_))) throw std::runtime_error("apply_state: states must be [ids][state_size]");
        ck(sb2_apply_state(h_, int64_t(ids.size()), ids.data(), states.data(), cids.data(), int(cids.size()), missing.data(), &n));
        missing.resize(size_t(n));
        return missing;
    }
    // :626-637; q_adjust_result of core/model_state_tuning.h:11-16
    q_adjust_result adjust_state_to_target_flow(double wanted_flow_m3s, const std::vector<int64_t>& cids, size_t start_step = 0, double scale_range = 3.0,
                                                double scale_eps = 1e-3, size_t max_iter = 300, size_t n_steps = 1) {
        sb2_q_adjust_result r{};
        ck(sb2_adjust_state_to_target_flow(h_, wanted_flow_m3s, cids.data(), int(cids.size()), int64_t(start_step), scale_range, scale_eps,
                                           int64_t(max_iter), int64_t(n_steps), &r));
        return q_adjust_result{r.q_0, r.q_r, std::string(r.diagnostics)};
    }

    void initialize_cell_environment(const fixed_dt& ta) { ck(sb2_initialize_cell_environment(h_, ta.t, ta.dt, int64_t(ta.n))); time_axis = ta; }  // :359-364
    bool interpolate(const interpolation_parameter& ip, const region_environment& env, bool best_effort = true) {                                   // :397-527
        for (int v = 0; v < SB2_N_FORCING; ++v) {
            const geo_point_sources& s = env.of(v);
            // the C ABI takes no element counts: a mis-shaped vector would be over-read during the upload
            if (s.xyz.size() % 3 != 0) throw std::runtime_error("interpolate: source xyz must be [n_sources][3]");
            if (s.values.size() != time_axis.n * s.size()) throw std::runtime_error("interpolate: source values must be [n_steps][n_sources]");
            ck(sb2_set_sources(h_, v, int64_t(s.size()), s.size() ? s.xyz.data() : nullptr, s.size() ? s.values.data() : nullptr));
        }
        int ok = 0;
        ck(sb2_interpolate(h_, &ip, best_effort ? 1 : 0, &ok));
        ip_parameter = ip;
        return ok != 0;
    }
    // a variable's series on their own point axis (any resolution), projected onto the model axis on the device (:426-438)
    void set_sources_on_axis(int var, const std::vector<double>& xyz, const std::vector<int64_t>& t_us, int64_t t_end_us,
                             const std::vector<double>& values /* [points][sources] */, int point_interpretation) {
        if (xyz.size() % 3 != 0 || values.size() != t_us.size() * (xyz.size() / 3))
            throw std::runtime_error("set_sources_on_axis: xyz must be [n_sources][3] and values [n_points][n_sources]");
        ck(sb2_set_sources_on_axis(h_, var, int64_t(xyz.size() / 3), xyz.data(), int64_t(t_us.size()), t_us.data(), t_end_us, values.data(),
                                   point_interpretation));
    }
    bool run_interpolation(const interpolation_parameter& ip, const fixed_dt& ta, const region_environment& env, bool best_effort = true) {         // :546-549
        initialize_cell_environment(ta);
        return interpolate(ip, env, best_effort);
    }
    bool is_cell_env_ts_ok() { int ok = 0; ck(sb2_is_cell_env_ts_ok(h_, &ok)); return ok != 0; }                                                  // :954-962

    void run_cells(size_t /*use_ncore*/ = 0, int start_step = 0, int n_steps = 0) { ck(sb2_run_cells(h_, start_step, n_steps)); }                   // :578-597

    // forcing ensemble (sb2_run_ensemble): every member's interpolation + run_cells(start_step, n_steps) from the current state in one
    // pass; per variable every member gives stations (the same positions) or none does (the model's own sources serve all members).
    // -> discharge and charge [member][cix][step], as catchment_discharges; the model is left as it was
    struct ensemble_result { std::vector<std::vector<std::vector<double>>> discharge, charge; };
    ensemble_result run_ensemble(const interpolation_parameter& ip, const std::vector<region_environment>& members, int start_step = 0,
                                 int n_steps = 0, int window_steps = 4096) {
        static const char* names[SB2_N_FORCING] = {"temperature", "precipitation", "radiation", "wind_speed", "rel_hum"};
        const size_t E = members.size();
        if (E == 0) throw std::runtime_error("run_ensemble: no members");
        for (int v = 0; v < SB2_N_FORCING; ++v) ck(sb2_set_ensemble_sources(h_, v, 0, 0, nullptr, nullptr));  // the member counts must agree
        for (int v = 0; v < SB2_N_FORCING; ++v) {
            const geo_point_sources& s0 = members[0].of(v);
            std::vector<double> values;
            for (const region_environment& env : members) {
                const geo_point_sources& s = env.of(v);
                // as interpolate: the C ABI takes no element counts, so a mis-shaped vector is refused here
                if (s.xyz != s0.xyz || s.xyz.size() % 3 != 0 || s.values.size() != time_axis.n * s.size())
                    throw std::runtime_error(std::string("run_ensemble: ") + names[v] +
                                             ": every member needs the same source positions [n_sources][3] and values [n_steps][n_sources]");
                values.insert(values.end(), s.values.begin(), s.values.end());
            }
            ck(sb2_set_ensemble_sources(h_, v, s0.size() ? int64_t(E) : 0, int64_t(s0.size()), s0.size() ? s0.xyz.data() : nullptr,
                                        s0.size() ? values.data() : nullptr));
        }
        const size_t count = n_steps > 0 ? size_t(n_steps) : time_axis.n, nc = number_of_catchments();
        std::vector<double> q(E * count * nc), c(q.size());
        ck(sb2_run_ensemble(h_, &ip, start_step, n_steps, window_steps, q.data(), c.data()));
        ip_parameter = ip;
        ensemble_result r;
        for (auto* out : {&r.discharge, &r.charge}) out->assign(E, std::vector<std::vector<double>>(nc, std::vector<double>(count)));
        for (size_t e = 0; e < E; ++e)
            for (size_t t = 0; t < count; ++t)
                for (size_t k = 0; k < nc; ++k) {
                    r.discharge[e][k][t] = q[(e * count + t) * nc + k];
                    r.charge[e][k][t] = c[(e * count + t) * nc + k];
                }
        return r;
    }

    // catchment_discharges(TSV&) (:873-885): cr[cix] = the catchment's series over the whole axis
    void catchment_discharges(std::vector<std::vector<double>>& cr) const { fetch(cr, sb2_catchment_discharges); }
    void catchment_charges(std::vector<std::vector<double>>& cr) const { fetch(cr, sb2_catchment_charges); }
    // cell.rc.<series> of every cell, [step][cell]
    std::vector<double> response(int series) const {
        std::vector<double> v(time_axis.n * size());
        ck(sb2_get_response(h_, series, 0, int64_t(time_axis.n), v.data(), SB2_TIME_MAJOR));
        return v;
    }
    // statistics readers (api/api.h:178-1600 over core/cell_model.h:194-406): kind / series / op / scope are the SB2_STAT_* / SB2_SCOPE_*
    // constants, e.g. basic_cell_statistics::discharge(cids) = statistics(SB2_STAT_RESPONSE, SB2_R_AVG_DISCHARGE, cids, SB2_STAT_SUM)
    std::vector<double> statistics(int kind, int series, const std::vector<int64_t>& indexes, int op, int scope = SB2_SCOPE_CATCHMENT_IX) const {
        std::vector<double> v(time_axis.n + ((kind == SB2_STAT_STATE || kind == SB2_STAT_AE_POT_RATIO) ? 1 : 0));
        ck(sb2_statistics_series(h_, kind, series, indexes.data(), int(indexes.size()), scope, op, 0, int64_t(v.size()), v.data()));
        return v;
    }
    double statistics_value(int kind, int series, const std::vector<int64_t>& indexes, size_t ith_timestep, int op,
                            int scope = SB2_SCOPE_CATCHMENT_IX) const {
        double v = 0.0;
        ck(sb2_statistics_series(h_, kind, series, indexes.data(), int(indexes.size()), scope, op == SB2_STAT_AREA_AVERAGE ? SB2_STAT_AREA_AVERAGE_VALUE : op,
                                 int64_t(ith_timestep), 1, &v));
        return v;
    }
    std::vector<double> statistics_cells(int kind, int series, const std::vector<int64_t>& indexes, size_t ith_timestep,
                                         int scope = SB2_SCOPE_CATCHMENT_IX) const {
        std::vector<double> v(size());
        int64_t n = 0;
        ck(sb2_statistics_cells(h_, kind, series, indexes.data(), int(indexes.size()), scope, int64_t(ith_timestep), v.data(), &n));
        v.resize(size_t(n));
        return v;
    }
    std::vector<double> river_output_flow_m3s(int64_t rid) { std::vector<double> v(time_axis.n); ck(sb2_river_flows(h_, rid, 0, int64_t(time_axis.n), nullptr, nullptr, v.data())); return v; }  // :926-933
    void set_river_network(const std::vector<double>& rivers6) {
        if (rivers6.size() % 6 != 0) throw std::runtime_error("set_river_network: rivers must be [n][6]");
        ck(sb2_set_river_network(h_, int64_t(rivers6.size() / 6), rivers6.data()));
    }

  private:
    template <class F>
    void fetch(std::vector<std::vector<double>>& cr, F f) const {
        const size_t nc = number_of_catchments(), T = time_axis.n;
        std::vector<double> flat(T * nc);
        ck(f(h_, 0, int64_t(T), flat.data()));
        cr.assign(nc, std::vector<double>(T));
        for (size_t t = 0; t < T; ++t)
            for (size_t k = 0; k < nc; ++k) cr[k][t] = flat[t * nc + k];
    }
};

// ---- model_calibration (core/model_calibration.h:242-329, 404-900; api/boostpython/expose.h:472-731) -------------------------------
// target_specification<PS>: the observed series on its own axis and what of the model it is compared with.  The axis is fixed_dt
// (t0_us, dt_us), or a point axis given by its n + 1 period boundaries (time_axis::point_dt); a CALENDAR axis (time_axis::calendar_dt:
// months, years, ... ) is taken by expanding it into those boundaries with calendar_period_points().
enum target_spec_calc_type { NASH_SUTCLIFFE = 0, KLING_GUPTA = 1, ABS_DIFF = 2, RMSE = 3 };
enum target_property_type { DISCHARGE = 0, SNOW_COVERED_AREA = 1, SNOW_WATER_EQUIVALENT = 2, ROUTED_DISCHARGE = 3, CELL_CHARGE = 4 };
struct target_specification {
    std::vector<double> values;
    utctime t0_us = 0;
    utctimespan dt_us = 0;
    std::vector<int64_t> catchment_indexes;
    double scale_factor = 1.0;
    int calc_mode = NASH_SUTCLIFFE, catchment_property = DISCHARGE;
    double s_r = 1.0, s_a = 1.0, s_b = 1.0;
    int64_t river_id = 0;
    std::string uid;
    std::vector<utctime> period_points_us;  // empty: the fixed_dt axis above
};
enum calendar_unit { CAL_DAY, CAL_WEEK, CAL_MONTH, CAL_QUARTER, CAL_YEAR };
// n + 1 boundaries of n calendar periods from t0 (UTC calendar, core/utctime_utilities.cpp:151-228: calendar::add with month / year
// arithmetic on the civil date, the day of month clipped to the target month's length)
inline std::vector<utctime> calendar_period_points(utctime t0_us, calendar_unit unit, size_t n) {
    const int64_t day = 86400LL * 1000000LL;
    auto civil = [](int64_t z, int64_t& y, unsigned& m, unsigned& d) {  // days since 1970-01-01 -> y-m-d (proleptic Gregorian)
        z += 719468;
        const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
        const unsigned doe = unsigned(z - era * 146097);
        const unsigned yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
        y = int64_t(yoe) + era * 400;
        const unsigned doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
        const unsigned mp = (5 * doy + 2) / 153;
        d = doy - (153 * mp + 2) / 5 + 1;
        m = mp < 10 ? mp + 3 : mp - 9;
        y += m <= 2;
    };
    auto days = [](int64_t y, unsigned m, unsigned d) {
        y -= m <= 2;
        const int64_t era = (y >= 0 ? y : y - 399) / 400;
        const unsigned yoe = unsigned(y - era * 400);
        const unsigned doy = (153 * (m > 2 ? m - 3 : m + 9) + 2) / 5 + d - 1;
        const unsigned doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
        return era * 146097 + int64_t(doe) - 719468;
    };
    std::vector<utctime> pts(n + 1);
    const int64_t d0 = t0_us >= 0 ? t0_us / day : -((-t0_us + day - 1) / day), tod = t0_us - d0 * day;
    int64_t y; unsigned m, d;
    civil(d0, y, m, d);
    for (size_t i = 0; i <= n; ++i) {
        if (unit == CAL_DAY || unit == CAL_WEEK) { pts[i] = t0_us + int64_t(i) * (unit == CAL_DAY ? day : 7 * day); continue; }
        const int64_t months = int64_t(i) * (unit == CAL_MONTH ? 1 : unit == CAL_QUARTER ? 3 : 12);
        const int64_t mm = int64_t(m) - 1 + months;
        const int64_t yy = y + (mm >= 0 ? mm / 12 : -((-mm + 11) / 12));
        const unsigned mo = unsigned(mm - (yy - y) * 12) + 1;
        static const unsigned mdays[12] = {31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
        const bool leap = (yy % 4 == 0 && yy % 100 != 0) || yy % 400 == 0;
        const unsigned last = mdays[mo - 1] + ((mo == 2 && leap) ? 1 : 0);
        pts[i] = days(yy, mo, d > last ? last : d) * day + tod;
    }
    return pts;
}

// optimizer<M, PA, PS> (:404-900): the goal-function entry runs on the device (sb2_calculate_goal_function, one parameter set; and
// sb2_calculate_goal_function_batch, a whole population as grid layers of the step kernels).  The search algorithms are host code in the
// reference too (dlib BOBYQA / global search, core/dream_optimizer.cpp, core/sceua_optimizer.cpp); dlib is not available here, and the
// drivers below are host-side stand-ins with the reference's signatures and meaning of the arguments -- NOT reproductions of those
// algorithms' random sequences: `optimize` is a bounded Nelder-Mead simplex in the scaled space (tr_start = initial simplex edge, tr_stop =
// simplex diameter to stop at), `optimize_dream` a differential-evolution Markov chain and `optimize_sceua` a shuffled complex evolution,
// both of which hand every generation's candidates to the device in ONE batch call.
template <int STACK>
class optimizer {
  public:
    using region_model_t = region_model<STACK>;
    using parameter_t = std::vector<double>;
    parameter_t parameter_lower_bound, parameter_upper_bound;
    std::vector<parameter_t> parameters_trace;
    std::vector<double> goal_fn_trace;
    std::vector<target_specification> targets;
    region_model_t& model;
    size_t n_single_calls = 0, n_batch_calls = 0;  // device entries used so far (diagnostic)

    explicit optimizer(region_model_t& m) : model(m) {}
    optimizer(region_model_t& m, const std::vector<target_specification>& t, const parameter_t& p_min, const parameter_t& p_max) : model(m) {
        set_target_specification(t, p_min, p_max);
    }
    void set_target_specification(const std::vector<target_specification>& t, const parameter_t& p_min, const parameter_t& p_max) {  // :575-589
        set_parameter_ranges(p_min, p_max);
        targets = t;
        std::vector<sb2_target> a(t.size());
        for (size_t i = 0; i < t.size(); ++i) {
            const target_specification& s = targets[i];
            if (!s.period_points_us.empty() && s.period_points_us.size() != s.values.size() + 1)
                throw std::runtime_error("target_specification: a point axis needs one more boundary than values");
            a[i].values = s.values.data(); a[i].t0_us = s.t0_us; a[i].dt_us = s.dt_us; a[i].n = int64_t(s.values.size());
            a[i].catchment_ids = s.catchment_indexes.data(); a[i].n_catchments = int32_t(s.catchment_indexes.size());
            a[i].river_id = s.river_id; a[i].scale_factor = s.scale_factor; a[i].calc_mode = s.calc_mode; a[i].property = s.catchment_property;
            a[i].s_r = s.s_r; a[i].s_a = s.s_a; a[i].s_b = s.s_b;
            a[i].period_points_us = s.period_points_us.empty() ? nullptr : s.period_points_us.data();
        }
        ck(sb2_set_targets(model.handle(), int(a.size()), a.data()));
    }
    void set_parameter_ranges(const parameter_t& p_min, const parameter_t& p_max) {  // :591-600
        const size_t n = size_t(sb2_parameter_size(model.handle()));
        if (p_min.size() != n || p_max.size() != n) throw std::runtime_error("p_min and p_max must have parameter size");
        parameter_lower_bound = p_min;
        parameter_upper_bound = p_max;
    }
    bool active_parameter(size_t i) const { return std::fabs(parameter_upper_bound[i] - parameter_lower_bound[i]) > 0.000001; }  // :424
    void set_verbose_level(int level) { verbose_ = level; }                                                                    // :683
    void reset_states() { model.revert_to_initial_state(); }                                                                   // :674-678
    size_t trace_size() const { return goal_fn_trace.size(); }
    double trace_goal_function_value(size_t i) const { return goal_fn_trace.at(i); }
    parameter_t trace_parameter(size_t i) const { return parameters_trace.at(i); }

    double calculate_goal_function(const parameter_t& p) {  // :691-699
        double g = 0.0;
        ck(sb2_calculate_goal_function(model.handle(), p.data(), int(p.size()), &g));
        ++n_single_calls;
        trace(p, g);
        return g;
    }
    // a population [n_sets][parameter_size] in one device pass; the values equal n_sets calls of calculate_goal_function
    std::vector<double> calculate_goal_function_batch(const std::vector<parameter_t>& P) {
        const size_t n = size_t(sb2_parameter_size(model.handle()));
        std::vector<double> flat(P.size() * n), g(P.size());
        for (size_t k = 0; k < P.size(); ++k) {
            if (P[k].size() != n) throw std::runtime_error("calculate_goal_function_batch: every parameter set must have parameter size");
            std::copy(P[k].begin(), P[k].end(), flat.begin() + k * n);
        }
        if (!P.empty()) ck(sb2_calculate_goal_function_batch(model.handle(), int64_t(P.size()), flat.data(), g.data()));
        ++n_batch_calls;
        for (size_t k = 0; k < P.size(); ++k) trace(P[k], g[k]);
        return g;
    }

    // local search from p (signature of optimize(p, max_n_evaluations, tr_start, tr_stop), :602-633)
    parameter_t optimize(const parameter_t& p, size_t max_n_evaluations, double tr_start, double tr_stop) {
        begin(p);
        const size_t d = act_.size();
        if (d == 0) return p;
        std::vector<std::vector<double>> x(d + 1, scaled(p));
        for (size_t i = 0; i < d; ++i) x[i + 1][i] = x[i + 1][i] + tr_start <= 1.0 ? x[i + 1][i] + tr_start : x[i + 1][i] - tr_start;
        std::vector<double> f = eval(x);
        size_t evals = d + 1;
        while (evals < max_n_evaluations) {
            std::vector<size_t> o(d + 1);
            for (size_t i = 0; i <= d; ++i) o[i] = i;
            std::sort(o.begin(), o.end(), [&](size_t a, size_t b) { return f[a] < f[b]; });
            double diam = 0.0;
            for (size_t i = 1; i <= d; ++i)
                for (size_t j = 0; j < d; ++j) diam = std::max(diam, std::fabs(x[o[i]][j] - x[o[0]][j]));
            if (diam < tr_stop) break;
            std::vector<double> c(d, 0.0);
            for (size_t i = 0; i < d; ++i)
                for (size_t j = 0; j < d; ++j) c[j] += x[o[i]][j] / double(d);
            const size_t w = o[d];
            auto along = [&](double t) { std::vector<double> y(d); for (size_t j = 0; j < d; ++j) y[j] = clip(c[j] + t * (x[w][j] - c[j])); return y; };
            // reflection, expansion and both contractions in one device pass (four candidates; the simplex logic picks among them)
            std::vector<std::vector<double>> cand{along(-1.0), along(-2.0), along(-0.5), along(0.5)};
            const std::vector<double> fc = eval(cand);
            evals += 4;
            const double f_best = f[o[0]], f_second_worst = f[o[d - 1]];
            if (fc[0] < f_best && fc[1] < fc[0]) { x[w] = cand[1]; f[w] = fc[1]; }
            else if (fc[0] < f_second_worst) { x[w] = cand[0]; f[w] = fc[0]; }
            else if (fc[0] < f[w] && fc[2] <= fc[0]) { x[w] = cand[2]; f[w] = fc[2]; }
            else if (fc[3] < f[w]) { x[w] = cand[3]; f[w] = fc[3]; }
            else {  // shrink towards the best vertex
                std::vector<std::vector<double>> sh;
                for (size_t i = 1; i <= d; ++i) { for (size_t j = 0; j < d; ++j) x[o[i]][j] = x[o[0]][j] + 0.5 * (x[o[i]][j] - x[o[0]][j]); sh.push_back(x[o[i]]); }
                const std::vector<double> fs = eval(sh);
                for (size_t i = 1; i <= d; ++i) f[o[i]] = fs[i - 1];
                evals += d;
            }
        }
        return expanded(x[size_t(std::min_element(f.begin(), f.end()) - f.begin())]);
    }
    // population search (signature of optimize_dream(p, max_n_evaluations), :652-668): differential-evolution Markov chain, one batch per generation
    parameter_t optimize_dream(const parameter_t& p, size_t max_n_evaluations) {
        begin(p);
        const size_t d = act_.size();
        if (d == 0) return p;
        const size_t N = std::max<size_t>(2 * d, 8);
        std::vector<std::vector<double>> x(N, std::vector<double>(d));
        x[0] = scaled(p);
        for (size_t i = 1; i < N; ++i) for (size_t j = 0; j < d; ++j) x[i][j] = uni_();
        std::vector<double> f = eval(x);
        size_t evals = N;
        const double gamma = 2.38 / std::sqrt(2.0 * double(d));
        while (evals + N <= max_n_evaluations) {
            std::vector<std::vector<double>> y(N, std::vector<double>(d));
            for (size_t i = 0; i < N; ++i) {
                size_t a = i, b = i;
                while (a == i) a = size_t(uni_() * double(N)) % N;
                while (b == i || b == a) b = size_t(uni_() * double(N)) % N;
                const double g = (uni_() < 0.1) ? 1.0 : gamma;  // every tenth proposal jumps between modes
                for (size_t j = 0; j < d; ++j) y[i][j] = reflect(x[i][j] + g * (x[a][j] - x[b][j]) + 1e-4 * (uni_() - 0.5));
            }
            const std::vector<double> fy = eval(y);  // the whole generation in ONE device pass
            evals += N;
            for (size_t i = 0; i < N; ++i)
                if (fy[i] <= f[i] || uni_() < std::exp(-(fy[i] - f[i]) / temperature_)) { x[i] = y[i]; f[i] = fy[i]; }
        }
        return best_of_trace();
    }
    // population search (signature of optimize_sceua(p, max_n_evaluations, x_eps, y_eps), :670-672): shuffled complex evolution
    // (Duan, Sorooshian, Gupta 1994), the complexes evolve in lock step so that each of their moves is one batch
    parameter_t optimize_sceua(const parameter_t& p, size_t max_n_evaluations, double x_eps, double y_eps) {
        begin(p);
        const size_t d = act_.size();
        if (d == 0) return p;
        const size_t m = 2 * d + 1, q = d + 1, n_cx = 2, s = m * n_cx;
        std::vector<std::vector<double>> x(s, std::vector<double>(d));
        x[0] = scaled(p);
        for (size_t i = 1; i < s; ++i) for (size_t j = 0; j < d; ++j) x[i][j] = uni_();
        std::vector<double> f = eval(x);
        size_t evals = s;
        double last_best = std::numeric_limits<double>::infinity();
        while (evals < max_n_evaluations) {
            std::vector<size_t> o(s);
            for (size_t i = 0; i < s; ++i) o[i] = i;
            std::sort(o.begin(), o.end(), [&](size_t a, size_t b) { return f[a] < f[b]; });
            double range = 0.0;
            for (size_t j = 0; j < d; ++j) {
                double lo = 1.0, hi = 0.0;
                for (size_t i = 0; i < s; ++i) { lo = std::min(lo, x[i][j]); hi = std::max(hi, x[i][j]); }
                range = std::max(range, hi - lo);
            }
            if (range < x_eps || std::fabs(last_best - f[o[0]]) < y_eps) break;
            last_best = f[o[0]];
            for (size_t step = 0; step < m && evals < max_n_evaluations; ++step) {  // beta = m evolution steps per shuffle
                std::vector<std::vector<size_t>> sub(n_cx);
                std::vector<std::vector<double>> refl(n_cx), contr(n_cx), mut(n_cx);
                for (size_t k = 0; k < n_cx; ++k) {  // complex k = every n_cx-th point of the ranking; q of its points, triangular preference
                    std::vector<size_t> cx;
                    for (size_t i = k; i < s; i += n_cx) cx.push_back(o[i]);
                    std::sort(cx.begin(), cx.end(), [&](size_t a, size_t b) { return f[a] < f[b]; });
                    std::vector<size_t> pick;
                    while (pick.size() < q) {
                        const size_t r = size_t(double(m) + 0.5 - std::sqrt((double(m) + 0.5) * (double(m) + 0.5) - double(m) * double(m + 1) * uni_()));
                        const size_t c = cx[std::min(r, m - 1)];
                        if (std::find(pick.begin(), pick.end(), c) == pick.end()) pick.push_back(c);
                    }
                    std::sort(pick.begin(), pick.end(), [&](size_t a, size_t b) { return f[a] < f[b]; });
                    sub[k] = pick;
                    std::vector<double> g(d, 0.0);
                    for (size_t i = 0; i + 1 < q; ++i) for (size_t j = 0; j < d; ++j) g[j] += x[pick[i]][j] / double(q - 1);
                    const std::vector<double>& w = x[pick[q - 1]];
                    refl[k].resize(d); contr[k].resize(d); mut[k].resize(d);
                    bool inside = true;
                    for (size_t j = 0; j < d; ++j) {
                        refl[k][j] = 2.0 * g[j] - w[j];
                        inside = inside && refl[k][j] >= 0.0 && refl[k][j] <= 1.0;
                        contr[k][j] = 0.5 * (g[j] + w[j]);
                        mut[k][j] = uni_();
                    }
                    if (!inside) refl[k] = mut[k];
                }
                std::vector<std::vector<double>> cand;
                for (size_t k = 0; k < n_cx; ++k) { cand.push_back(refl[k]); cand.push_back(contr[k]); cand.push_back(mut[k]); }
                const std::vector<double> fc = eval(cand);  // reflection, contraction and mutation points of every complex in ONE device pass
                evals += cand.size();
                for (size_t k = 0; k < n_cx; ++k) {
                    const size_t w = sub[k][q - 1];
                    if (fc[3 * k] < f[w]) { x[w] = refl[k]; f[w] = fc[3 * k]; }
                    else if (fc[3 * k + 1] < f[w]) { x[w] = contr[k]; f[w] = fc[3 * k + 1]; }
                    else { x[w] = mut[k]; f[w] = fc[3 * k + 2]; }
                }
            }
        }
        return best_of_trace();
    }

  private:
    void ck(int rc) const { if (rc != 0) throw std::runtime_error(sb2_last_error(model.handle())); }
    int verbose_ = 0;
    double temperature_ = 0.01;  // acceptance scale of the Markov chain, in units of the goal function
    std::vector<size_t> act_;
    parameter_t p_full_;
    uint64_t rng_ = 0x9E3779B97F4A7C15ULL;
    double uni_() {  // xorshift64*: deterministic search sequences
        rng_ ^= rng_ >> 12; rng_ ^= rng_ << 25; rng_ ^= rng_ >> 27;
        return double((rng_ * 0x2545F4914F6CDD1DULL) >> 11) * (1.0 / 9007199254740992.0);
    }
    static double clip(double v) { return v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v); }
    static double reflect(double v) { while (v < 0.0 || v > 1.0) v = v < 0.0 ? -v : 2.0 - v; return v; }
    void trace(const parameter_t& p, double g) {
        parameters_trace.push_back(p);
        goal_fn_trace.push_back(g);
        if (verbose_ > 0) std::printf("goal %zu: %.10g\n", goal_fn_trace.size(), g);
    }
    void begin(const parameter_t& p) {
        if (parameter_lower_bound.size() != p.size()) throw std::runtime_error("optimize: parameter ranges are not set");
        p_full_ = p;
        act_.clear();
        for (size_t i = 0; i < p.size(); ++i)
            if (active_parameter(i)) act_.push_back(i);
        rng_ = 0x9E3779B97F4A7C15ULL;
    }
    std::vector<double> scaled(const parameter_t& p) const {  // active parameters in [0, 1] (:435-453, 707-739)
        std::vector<double> x(act_.size());
        for (size_t k = 0; k < act_.size(); ++k) {
            const size_t i = act_[k];
            x[k] = clip((p[i] - parameter_lower_bound[i]) / (parameter_upper_bound[i] - parameter_lower_bound[i]));
        }
        return x;
    }
    parameter_t expanded(const std::vector<double>& x) const {
        parameter_t p = p_full_;
        for (size_t k = 0; k < act_.size(); ++k) {
            const size_t i = act_[k];
            p[i] = parameter_lower_bound[i] + x[k] * (parameter_upper_bound[i] - parameter_lower_bound[i]);
        }
        return p;
    }
    std::vector<double> eval(const std::vector<std::vector<double>>& xs) {
        std::vector<parameter_t> P;
        for (auto& x : xs) P.push_back(expanded(x));
        return calculate_goal_function_batch(P);
    }
    parameter_t best_of_trace() const {
        return parameters_trace[size_t(std::min_element(goal_fn_trace.begin(), goal_fn_trace.end()) - goal_fn_trace.begin())];
    }
};

using pt_gs_k_region_model = region_model<SB2_PT_GS_K>;
using pt_hs_k_region_model = region_model<SB2_PT_HS_K>;
using hbv_stack_region_model = region_model<SB2_HBV_STACK>;
using pt_ss_k_region_model = region_model<SB2_PT_SS_K>;
using pt_hps_k_region_model = region_model<SB2_PT_HPS_K>;

}  // namespace shyft_b200
