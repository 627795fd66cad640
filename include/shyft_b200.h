/* ============================================================================
 * shyft_b200.h -- C ABI of the B200-native region-model hot path.
 *
 * The reference (magneano/shyft, VERSION 1675) has no FFI for this path: Python reaches the C++
 * template members of region_model<cell_t> through boost.python (api/boostpython/expose.h:143-430).
 * This header is the boundary a maintainer binds instead; each entry point cites the reference
 * member it stands in for (paths relative to the reference root).  Plain pointers and sizes only,
 * no exceptions cross it: every call returns 0 on success, non-zero on failure, and
 * sb2_last_error() then returns the message (the reference's std::runtime_error text where one
 * exists).  Host buffers are caller-owned; device buffers are library-owned unless a *_device
 * variant says otherwise.  A model is not safe for concurrent calls (neither is the reference's,
 * core/model_calibration.h:832); distinct models are independent.
 * ==========================================================================*/
#ifndef SHYFT_B200_H
#define SHYFT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb2_model sb2_model;

/* method stacks (core/pt_gs_k.h, core/pt_hs_k.h, core/hbv_stack.h, core/pt_ss_k.h, core/pt_hps_k.h) */
enum { SB2_PT_GS_K = 0, SB2_PT_HS_K = 1, SB2_HBV_STACK = 2, SB2_PT_SS_K = 3, SB2_PT_HPS_K = 4 };
/* forcing variables, the members of cell.env_ts (core/cell_model.h:47-56) */
enum { SB2_TEMPERATURE = 0, SB2_PRECIPITATION = 1, SB2_RADIATION = 2, SB2_WIND_SPEED = 3, SB2_REL_HUM = 4, SB2_N_FORCING = 5 };
/* host array layouts for [time x cell] data */
enum { SB2_TIME_MAJOR = 0 /* [t][cell] */, SB2_CELL_MAJOR = 1 /* [cell][t], the reference's per-cell vector<double> */ };

/* response collector bits (core/pt_gs_k_cell_model.h:41-131): which per-cell series run_cells keeps */
enum {
    SB2_COLLECT_NONE = 0,          /* catchment sums only (calibration inner loop)                               */
    SB2_COLLECT_DISCHARGE = 1,     /* discharge_collector: avg_discharge, charge_m3s                              */
    SB2_COLLECT_SNOW = 2,          /* + snow_sca, snow_swe (set_snow_sca_swe_collection)                          */
    SB2_COLLECT_ALL = 7,           /* all_response_collector: + snow_outflow, glacier_melt, ae_output, pe_output  */
    SB2_COLLECT_STATE = 8          /* state_collector (T+1 points per series), set_state_collection               */
};
/* per-cell response series ids (all_response_collector member order); SB2_R_SOIL_OUTFLOW is hbv_stack only */
enum { SB2_R_AVG_DISCHARGE = 0, SB2_R_CHARGE_M3S, SB2_R_SNOW_SCA, SB2_R_SNOW_SWE, SB2_R_SNOW_OUTFLOW, SB2_R_GLACIER_MELT,
       SB2_R_AE_OUTPUT, SB2_R_PE_OUTPUT, SB2_R_SOIL_OUTFLOW, SB2_N_RESPONSE };
/* pt_gs_k state series ids (state_collector member order, core/pt_gs_k_cell_model.h:146-208).
 * pt_hs_k: 0 kirchner_discharge, 1 snow_sca, 2 snow_swe, 3..7 sp[0..4], 8..12 sw[0..4] (core/pt_hs_k_cell_model.h:148-206);
 * hbv_stack: 0 snow_swe, 1 snow_sca, 2 soil_moisture, 3 tank_uz, 4 tank_lz, 5..9 sp[0..4], 10..14 sw[0..4]
 * (core/hbv_stack_cell_model.h:148-213); sp / sw = the snow pack and its liquid water per quantile bin (five bins);
 * pt_ss_k: 0 kirchner_discharge, 1 snow_swe, 2 snow_sca, 3 snow_alpha, 4 snow_nu, 5 snow_lwc, 6 snow_residual
 * (core/pt_ss_k_cell_model.h:148-199);
 * pt_hps_k: 0 kirchner_discharge, 1 snow_sca, 2 snow_swe, 3 surface_heat, 4..8 sp[0..4], 9..13 sw[0..4], 14..18 albedo[0..4],
 * 19..23 iso_pot_energy[0..4] (core/pt_hps_k_cell_model.h:150-230). */
enum { SB2_S_KIRCHNER_DISCHARGE = 0, SB2_S_GS_ALBEDO, SB2_S_GS_LWC, SB2_S_GS_SURFACE_HEAT, SB2_S_GS_ALPHA, SB2_S_GS_SDC_MELT_MEAN,
       SB2_S_GS_ACC_MELT, SB2_S_GS_ISO_POT_ENERGY, SB2_S_GS_TEMP_SWE, SB2_N_STATE_SERIES = 24 };
enum { SB2_S_PTHSK_SP0 = 3, SB2_S_PTHSK_SW0 = 8, SB2_S_HBV_SP0 = 5, SB2_S_HBV_SW0 = 10, SB2_S_PTHPSK_SP0 = 4, SB2_S_PTHPSK_SW0 = 9,
       SB2_S_PTHPSK_ALBEDO0 = 14, SB2_S_PTHPSK_ISO0 = 19 };

/* geo_cell_data (core/geo_cell_data.h:107-138) flattened; one per cell, in the caller's cell order */
typedef struct sb2_geo_cell {
    double x, y, z;                 /* mid_point */
    double area;                    /* m2 */
    int64_t catchment_id;
    double radiation_slope_factor;
    double glacier, lake, reservoir, forest; /* land_type_fractions */
    int64_t routing_id;             /* routing_info.id, 0 = none */
    double routing_distance;        /* routing_info.distance [m] */
} sb2_geo_cell;

/* inverse_distance::parameter / temperature_parameter / precipitation_parameter (core/inverse_distance.h:38-74) */
typedef struct sb2_idw_parameter {
    int64_t max_members;
    double max_distance;
    double distance_measure_factor;
    double zscale;
    double default_temp_gradient;   /* temperature only */
    int32_t gradient_by_equation;   /* temperature only */
    double scale_factor;            /* precipitation only */
} sb2_idw_parameter;
/* bayesian_kriging::parameter (core/bayesian_kriging.h:204-230) */
typedef struct sb2_btk_parameter {
    double gradient_sd, sill, nug, range, zscale;
} sb2_btk_parameter;
/* interpolation_parameter (core/region_model.h:65-95) */
typedef struct sb2_interpolation_parameter {
    sb2_btk_parameter temperature;
    int32_t use_idw_for_temperature;
    sb2_idw_parameter temperature_idw;
    sb2_idw_parameter precipitation;
    sb2_idw_parameter wind_speed;
    sb2_idw_parameter radiation;
    sb2_idw_parameter rel_hum;
} sb2_interpolation_parameter;
void sb2_interpolation_parameter_default(sb2_interpolation_parameter* ip); /* the reference's default-constructed values */

/* ---- lifetime -------------------------------------------------------------------------------- */
/* region_model(const std::vector<geo_cell_data>&, const parameter_t&)  (core/region_model.h:283-291).
 * Assigns catchment_ix in order of first appearance of catchment_id (:233-249). `device` = CUDA ordinal. */
int sb2_model_create(int stack, int64_t n_cells, const sb2_geo_cell* cells, int device, sb2_model** out);
void sb2_model_destroy(sb2_model* m);
const char* sb2_last_error(const sb2_model* m); /* m == NULL: error of the last failed sb2_model_create on this thread */
int sb2_version(void);

int64_t sb2_size(const sb2_model* m);                                   /* region_model::size() :860 */
int64_t sb2_number_of_catchments(const sb2_model* m);                   /* :318 */
int sb2_catchment_ids(const sb2_model* m, int64_t* out);                /* cix -> cid, :320 */
int sb2_cell_catchment_ix(const sb2_model* m, int64_t* out);            /* geo.catchment_ix per cell */
int sb2_parameter_size(const sb2_model* m);                             /* parameter::size(): 31 / 18 / 22 */
int sb2_state_size(const sb2_model* m);                                 /* doubles per cell state: 9 / 13 / 15 (5 snow bins) */

/* ---- parameters, filter, state --------------------------------------------------------------- */
int sb2_set_region_parameter(sb2_model* m, const double* p, int n);                     /* :646-655, vector order of parameter::set */
int sb2_get_region_parameter(const sb2_model* m, double* p, int n);                     /* :660 */
int sb2_set_catchment_parameter(sb2_model* m, int64_t cid, const double* p, int n);     /* :668-678 */
int sb2_get_catchment_parameter(const sb2_model* m, int64_t cid, double* p, int n);     /* :702-708; the region parameter if no override */
int sb2_remove_catchment_parameter(sb2_model* m, int64_t cid);                          /* :683-691 */
int sb2_has_catchment_parameter(const sb2_model* m, int64_t cid);                       /* :693 */
int sb2_set_catchment_calculation_filter(sb2_model* m, const int64_t* cids, int n);     /* :715-729; n == 0 clears */
int sb2_set_states(sb2_model* m, const double* states, int64_t n_cells);                /* :802-809, [cell][state_size] */
int sb2_get_states(const sb2_model* m, double* states, int64_t n_cells);                /* :784-787 */
/* Flat state layouts ([cell][state_size], the order of the reference's state classes):
 *   pt_gs_k   9: gs.albedo, gs.lwc, gs.surface_heat, gs.alpha, gs.sdc_melt_mean, gs.acc_melt, gs.iso_pot_energy, gs.temp_swe, kirchner.q
 *   pt_hs_k  13: snow.swe, snow.sca, snow.sp[0..4], snow.sw[0..4], kirchner.q
 *   hbv_stack 15: snow.swe, snow.sca, snow.sp[0..4], snow.sw[0..4], soil.sm, tank.uz, tank.lz
 *   pt_ss_k   8: snow.nu, snow.alpha, snow.sca, snow.swe, snow.free_water, snow.residual, snow.num_units, kirchner.q
 *   pt_hps_k 24: hps.sp[0..4], hps.sw[0..4], hps.albedo[0..4], hps.iso_pot_energy[0..4], hps.surface_heat, hps.swe, hps.sca, kirchner.q
 * hbv_snow::state::distribute(parameter, false) (core/hbv_snow.h:114-118; called first thing by pt_hs_k::run :230 and run_hbv_stack :312):
 * rows whose ten snow bins are all zero -- the flat spelling of HbvSnowState(swe, sca) with empty bin vectors -- get sp / sw from swe, sca
 * and the cell's hs parameters (hbv_snow_common.h:44-67); other rows are left as they are.  Host side, in place, before sb2_set_states. */
int sb2_hbv_distribute_snow(const sb2_model* m, double* states, int64_t n_cells);
int sb2_set_initial_state(sb2_model* m, const double* states, int64_t n_cells);         /* the public member initial_state, :313 */
int sb2_get_initial_state(const sb2_model* m, double* states, int64_t n_cells);
int sb2_revert_to_initial_state(sb2_model* m);                                          /* :814-818 */
int sb2_adjust_q(sb2_model* m, double q_scale, const int64_t* cids, int n);             /* :831-837 */
/* Cell-identified state (api/api_state.h:34-148; `model.state.extract_state(cids)` / `.apply_state(states, cids)` in Python,
 * api/boostpython/expose.h:59-88).  cell_state_id_of (:58-60): (catchment id, (int)mid_point.x, (int)mid_point.y, (int)area).
 * extract: the states of the cells of `cids` (empty = all), in cell order, gathered on the device; ids / states hold up to sb2_size()
 * entries.  apply: every supplied state whose id.cid passes `cids` is written to the cell with the same id (among the cells of `cids`);
 * the positions of those that found no cell come back in `missing` (capacity n), exactly as state_io_handler::apply_state :119-140. */
typedef struct sb2_cell_state_id { int64_t cid, x, y, area; } sb2_cell_state_id;
int sb2_extract_state(const sb2_model* m, const int64_t* cids, int n_cids, sb2_cell_state_id* ids, double* states /* [.][state_size] */,
                      int64_t* n_out);
int sb2_apply_state(sb2_model* m, int64_t n, const sb2_cell_state_id* ids, const double* states /* [n][state_size] */, const int64_t* cids,
                    int n_cids, int64_t* missing, int64_t* n_missing);
int sb2_set_collector_mode(sb2_model* m, int collect_bits);                             /* cell type + set_state_collection / set_snow_sca_swe_collection :844-858 */
/* region_model::adjust_state_to_target_flow (:626-637) = adjust_state_model::tune_flow (core/model_state_tuning.h:38-118): scale the
 * ground storage of the cells of `cids` (empty = all) from the CURRENT state so that the mean avg_discharge of the n_steps steps from
 * start_step equals wanted_flow_m3s; the reference's q_adjust_result (:11-16) comes back by value.  On return the current state is the
 * adjusted one, the initial state and the catchment calculation filter are as before.  Needs a resident cell environment. */
typedef struct sb2_q_adjust_result {
    double q_0;             /* m3/s before the adjustment */
    double q_r;             /* m3/s reached */
    char diagnostics[512];  /* empty if ok */
} sb2_q_adjust_result;
int sb2_adjust_state_to_target_flow(sb2_model* m, double wanted_flow_m3s, const int64_t* cids, int n_cids, int64_t start_step,
                                    double scale_range /* 3.0 */, double scale_eps /* 1e-3 */, int64_t max_iter /* 300 */,
                                    int64_t n_steps /* 1 */, sb2_q_adjust_result* result);

/* ---- environment ------------------------------------------------------------------------------ */
/* initialize_cell_environment(time_axis) (:359-364): fixed_dt{t0, dt, n} in microseconds; env_ts reset to NaN */
int sb2_initialize_cell_environment(sb2_model* m, int64_t t0_us, int64_t dt_us, int64_t n);
/* write cell.env_ts.<var> directly (the "distributed series supplied by the orchestrator" case, :448-452) */
int sb2_set_cell_forcing(sb2_model* m, int var, const double* values, int layout);
int sb2_get_cell_forcing(const sb2_model* m, int var, int64_t start_step, int64_t n_steps, double* out, int layout);
/* region_environment sources (api/api.h:137-168): n_src geo-located series already on the model axis, values [t][src];
 * the identity resampling of average_accessor (core/time_series.h:2033-2072) is applied on upload */
int sb2_set_sources(sb2_model* m, int var, int64_t n_src, const double* xyz /* [src][3] */, const double* values /* [T][src] */);
/* The same for sources on their OWN point axis (any resolution; region_environment series are projected onto the model axis by
 * average_accessor<ts, timeaxis>, core/region_model.h:426-438 over core/time_series.h:202-310, 2033-2072): t_us [n_points] strictly
 * increasing point times shared by the n_src series, t_end_us = the series' total_period().end, values [n_points][n_src],
 * point_interpretation = the series' ts_point_fx.  The projection (true average per model step, NaN-aware, NaN from t_end on) runs
 * on the device. */
enum { SB2_POINT_AVERAGE_VALUE = 0 /* stair-case */, SB2_POINT_INSTANT_VALUE = 1 /* linear between points */ };
int sb2_set_sources_on_axis(sb2_model* m, int var, int64_t n_src, const double* xyz, int64_t n_points, const int64_t* t_us, int64_t t_end_us,
                            const double* values, int point_interpretation);
/* the sources of a variable as projected onto the model axis: out [T][n_src] */
/* ... and for sources that EACH bring their own point axis (every geo_point_ts of a region_environment owns its time-series,
 * api/api.h:137-168): source s has n_points[s] points, stored one source after the other in t_us / values (sum of n_points entries),
 * its own total-period end t_end_us[s] and point interpretation[s].  Projected on the device like the shared-axis form. */
int sb2_set_sources_on_axes(sb2_model* m, int var, int64_t n_src, const double* xyz /* [src][3] */, const int64_t* n_points /* [src] */,
                            const int64_t* t_us, const int64_t* t_end_us /* [src] */, const double* values,
                            const int32_t* point_interpretation /* [src] */);
int sb2_get_sources_on_model_axis(const sb2_model* m, int var, double* out);
/* interpolate(ip, env, best_effort) (:397-527) over the whole axis; returns 0 also when best_effort swallowed a
 * per-variable failure, in which case *all_ok (nullable) is 0 and that variable stays NaN */
int sb2_interpolate(sb2_model* m, const sb2_interpolation_parameter* ip, int best_effort, int* all_ok);
int sb2_is_cell_env_ts_ok(sb2_model* m, int* ok);                                       /* :954-962 */

/* ---- the hot path -------------------------------------------------------------------------------- */
/* run_cells(use_ncore, start_step, n_steps) (:578-597); same argument validation and messages; use_ncore has no
 * meaning on the device.  n_steps == 0 runs to the end of the axis. */
int sb2_run_cells(sb2_model* m, int start_step, int n_steps);
/* run_interpolation + run_cells window by window for axes whose [t][cell] forcing does not fit in HBM: each window
 * of `window_steps` steps is interpolated from the sources and stepped; per-cell series (if collected) hold the
 * last window only, catchment sums and states cover the whole call. */
int sb2_run_windowed(sb2_model* m, const sb2_interpolation_parameter* ip, int start_step, int n_steps, int window_steps);

/* ---- forcing ensembles ------------------------------------------------------------------------------ */
/* The members of a forecast ensemble (create_ensembles, shyft/orchestration/simulator.py) in one call instead of one
 * set_sources + interpolate + run_cells + catchment_discharges per member.  Member e of sb2_run_ensemble is bit for bit what that
 * loop gives: member e's stations set for every variable that has ensemble sources (the model's own sources for every other
 * variable), sb2_interpolate(ip, best_effort = 0), sb2_run_cells(start_step, n_steps) from the model's current state, and the
 * catchment sums of those rows.  The model is left as it was; initialize_cell_environment drops ensemble sources as it drops sources. */
/* one variable's stations for every member of a forcing ensemble, on the model axis: values [member][T][src] (as sb2_set_sources);
   n_members == 0 or n_src == 0 clears the variable's ensemble sources.  Every variable with ensemble sources has the same member count. */
int sb2_set_ensemble_sources(sb2_model* m, int var, int64_t n_members, int64_t n_src, const double* xyz, const double* values);
/* ... on one point axis shared by all members and stations: values [member][n_points][src] (as sb2_set_sources_on_axis) */
int sb2_set_ensemble_sources_on_axis(sb2_model* m, int var, int64_t n_members, int64_t n_src, const double* xyz, int64_t n_points,
                                     const int64_t* t_us, int64_t t_end_us, const double* values, int point_interpretation);
/* interpolate and step every member over [start_step, start_step + n_steps), window_steps at a time, from the model's current state
   (n_steps == 0: the whole axis); discharge and charge (nullable) [member][n_steps][n_catchments], cix order */
int sb2_run_ensemble(sb2_model* m, const sb2_interpolation_parameter* ip, int start_step, int n_steps, int window_steps,
                     double* discharge, double* charge);

/* ---- results ------------------------------------------------------------------------------------- */
/* cell.rc.<series> / cell.sc.<series> (api/boostpython/expose.h:98-120); out [n_steps][cell] or [cell][n_steps] */
int sb2_get_response(const sb2_model* m, int series, int64_t start_step, int64_t n_steps, double* out, int layout);
int sb2_get_state_series(const sb2_model* m, int series, int64_t start_step, int64_t n_points, double* out, int layout);
/* catchment_discharges / catchment_charges (:873-900): out [n_steps][n_catchments], cix order */
int sb2_catchment_discharges(const sb2_model* m, int64_t start_step, int64_t n_steps, double* out);
int sb2_catchment_charges(const sb2_model* m, int64_t start_step, int64_t n_steps, double* out);

/* ---- statistics readers over the resident series (core/cell_model.h:194-406 as used by api/api.h:178-1600) ------- */
/* which series: forcing variable (cell.env_ts), response series (cell.rc) or state series (cell.sc, instant values) */
enum { SB2_STAT_FORCING = 0, SB2_STAT_RESPONSE = 1, SB2_STAT_STATE = 2,
       SB2_STAT_AE_POT_RATIO = 3 /* series ignored: 1 - exp(-3 q / ae_scale_factor) of the instant Kirchner state, api/api.h:1519-1564 (pt_gs_k) */ };
/* stat_scope (core/cell_model.h:178-181): indexes are catchment ids or cell indexes; n_indexes == 0 selects every cell */
enum { SB2_SCOPE_CATCHMENT_IX = 0, SB2_SCOPE_CELL_IX = 1 };
enum { SB2_STAT_SUM = 0 /* sum_catchment_feature */, SB2_STAT_AREA_AVERAGE = 1 /* average_catchment_feature: r * (1/sum_area) */,
       SB2_STAT_AREA_AVERAGE_VALUE = 2 /* average_catchment_feature_value: r / sum_area */ };
/* sum_catchment_feature / average_catchment_feature (:230-268, :313-333): out [n_steps] (state series: points).  Errors as
 * verify_cids_exist (:197-213): "one or more supplied catchment_indexes does not exist:<cid>" / "Supplied cell index reference ..." */
int sb2_statistics_series(const sb2_model* m, int kind, int series, const int64_t* indexes, int n_indexes, int scope, int op,
                          int64_t start_step, int64_t n_steps, double* out);
/* catchment_feature (:381-402): the selected cells' values at one step, in cell order; *n_out = number written (<= size()) */
int sb2_statistics_cells(const sb2_model* m, int kind, int series, const int64_t* indexes, int n_indexes, int scope, int64_t step,
                         double* out, int64_t* n_out);
/* basic_cell_statistics geo sums (api/api.h:183-288): what = 0 total, 1 forest, 2 glacier, 3 lake, 4 reservoir, 5 unspecified,
 * 6 snow_storage area [m2], 7 area-weighted elevation [m] */
int sb2_statistics_geo(const sb2_model* m, int what, const int64_t* indexes, int n_indexes, int scope, double* out);

/* ---- routing (core/routing.h:145-383; region_model.h:909-949) -------------------------------------- */
/* river_network: rivers [n][6] = id, downstream id (0 = none), downstream distance [m], uhg velocity, alpha, beta (routing.h:98-123).
 * Validates ids and acyclicity like river_network::add / set_downstream_by_id (routing.h:160-250). */
int sb2_set_river_network(sb2_model* m, int64_t n_rivers, const double* rivers);
/* river_local_inflow_m3s / river_upstream_inflow_m3s / river_output_flow_m3s (region_model.h:926-949) of river `rid`
 * over [start_step, start_step+n_steps); any output pointer may be NULL.  Needs avg_discharge collected over the axis. */
int sb2_river_flows(sb2_model* m, int64_t rid, int64_t start_step, int64_t n_steps, double* local_inflow, double* upstream_inflow,
                    double* output);

/* ---- calibration: the goal-function entry (core/model_calibration.h:404-900) -------------------------- */
enum { SB2_GOAL_NASH_SUTCLIFFE = 0, SB2_GOAL_KLING_GUPTA = 1, SB2_GOAL_ABS_DIFF = 2, SB2_GOAL_RMSE = 3 };             /* target_spec_calc_type :217-222 */
enum { SB2_TARGET_DISCHARGE = 0, SB2_TARGET_SNOW_COVERED_AREA = 1, SB2_TARGET_SNOW_WATER_EQUIVALENT = 2,
       SB2_TARGET_ROUTED_DISCHARGE = 3, SB2_TARGET_CELL_CHARGE = 4 };                                                  /* target_property_type :225-231 */
/* target_specification (:242-329).  The target series lives on its own axis: fixed_dt {t0_us, dt_us, n} -- periods that are whole
 * runs of model steps are reduced in the goal kernel itself, any other fixed_dt axis is projected first -- or, when period_points_us
 * is set, a point axis of n periods [period_points_us[i], period_points_us[i+1]) (n + 1 strictly increasing times; time_axis::point_dt). */
typedef struct sb2_target {
    const double* values; int64_t t0_us, dt_us, n;
    const int64_t* catchment_ids; int32_t n_catchments;
    int64_t river_id;               /* ROUTED_DISCHARGE only */
    double scale_factor;
    int32_t calc_mode, property;
    double s_r, s_a, s_b;           /* Kling-Gupta weights */
    const int64_t* period_points_us; /* NULL: the fixed_dt axis above */
} sb2_target;
/* optimizer(model, targets, ...) + prepare_optimize (:517-552): stores the targets, switches snow collection on when a target
 * needs it, sets the calculation filter to the union of the target catchments, snapshots the initial state if unset. */
int sb2_set_targets(sb2_model* m, int n_targets, const sb2_target* targets);
/* optimizer::calculate_goal_function(full parameter vector) (:691-699) = run() (:830-899): set the region parameter, reset the
 * states, run_cells, evaluate every target, weighted mean. */
int sb2_calculate_goal_function(sb2_model* m, const double* p, int n, double* goal);
/* The same for n_sets parameter vectors P [n_sets][parameter_size] at once: the sets form an extra grid dimension of the cell
 * step kernel and share the forcing reads (the reference evaluates one set at a time, dream_optimizer.cpp:62,201). */
int sb2_calculate_goal_function_batch(sb2_model* m, int64_t n_sets, const double* P, double* goals);

/* ---- diagnostics ------------------------------------------------------------------------------------- */
/* Evaluate one device function on n rows of inputs (unit tests in the style of test/gamma_snow_test.cpp, test/kirchner_test.cpp):
 * fn 0 exp(x), 1 log(x), 2 pow(x,y), 3 lgamma(a), 4 gamma_p(a,x), 5 corr_lwc(z1,a1,b1,a2,b2), 6 calc_snow_state(shape,scale,y0,
 * lambda,lwd,max_water_frac,temp_swe) -> swe,sca, 7 kirchner step(c1,c2,c3,dt_hours,q,p,e) -> q,q_avg,ok.  Errors: sb2_last_error(NULL). */
int sb2_unit_eval(int device, int fn, int64_t n, const double* in, int n_in, double* out, int n_out);
/* Host-side algorithms of the library, callable without a device (CPU unit tests against the oracle): fn 0 the one-dimensional
 * minimiser of the state tuning (dlib find_min_single_variable restated, core/model_state_tuning.h:98-108) on
 * f(x) = (x - a)^2 + b cosh(x - c): in = a b c start begin end eps max_iter -> out = x f(x) evaluations failed(0/1);
 * fn 1 calendar: in = t_us -> day_of_year, seconds_of_year (core/utctime_utilities.cpp:230-255);
 * fn 2 make_uhg_from_gamma: in = n_steps alpha beta -> out[0] = length, out[1..] = weights (core/routing.h:399-421);
 * fn 3 unit-hydrograph steps: in = distance velocity dt_us -> n (core/routing.h:119-123, 326-330).  Returns 0 / 1 (bad arguments). */
int sb2_host_eval(int fn, const double* in, int n_in, double* out, int n_out);

/* IDW with all station values finite runs as a dense tensor-core contraction (results within ~1e-15 of the per-neighbour
 * weighted mean); on = 0 forces the per-neighbour kernel, which is bit-identical to the reference's operation order. */
int sb2_set_idw_dense(sb2_model* m, int on);

/* ---- device-side hooks (plumbing for torch.distributed / CUDA-event timing; not part of the reference surface) -- */
int sb2_set_stream(sb2_model* m, void* cuda_stream);           /* launch on this stream (default: the legacy default stream) */
int sb2_device_catchment_discharges(sb2_model* m, void** dptr, int64_t* n_steps, int64_t* n_catchments); /* [T][n_catch] fp64 in HBM */
int sb2_device_catchment_charges(sb2_model* m, void** dptr, int64_t* n_steps, int64_t* n_catchments);
/* diagnostic: with SB2_GUARD=1 in the environment every device buffer carries 4 KB red zones; -> number of buffers whose zones were
 * overwritten so far (0 = no out-of-bounds write seen), the first finding as text */
int64_t sb2_check_guards(char* message, int message_size);
int64_t sb2_kernel_launches(const sb2_model* m);               /* launches of this library's kernels since creation */
int sb2_step_chunk_steps(const sb2_model* m);                  /* steps one launch of the step kernels covers (0 before the first run) */
int sb2_last_run_kernel_ms(const sb2_model* m, float* step_ms, float* interp_ms); /* CUDA-event time of the last run's kernels */

#ifdef __cplusplus
}
#endif
#endif
