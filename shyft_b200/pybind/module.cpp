// pybind11 module over the C++ host shim (include/shyft_b200/region_model.hpp): the binding layer a maintainer puts where
// api/boostpython/expose.h:143-430 binds region_model<cell_t> today, with the class names the reference exposes to Python
// (PTGSKModel / PTGSKOptModel, PTHSKModel / PTHSKOptModel, HbvModel / HbvOptModel; shyft/api/<stack>/__init__.py).  SURVEY 8f item 2.
// boost.python itself cannot be built here, so this is pybind11; every numeric call goes shim -> C ABI -> CUDA library.
// numpy in, numpy out: geo cells as the 96-byte sb2_geo_cell records, states [cell][state_size], series [step][...].
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <memory>

#include <shyft_b200/region_model.hpp>

namespace py = pybind11;
namespace sb = shyft_b200;
using darray = py::array_t<double, py::array::c_style | py::array::forcecast>;

namespace {

std::vector<double> flat(const darray& a) { return std::vector<double>(a.data(), a.data() + a.size()); }

std::vector<sb::geo_cell_data> geo_vector(const py::array& a) {
    const py::buffer_info b = a.request();
    if (b.itemsize != py::ssize_t(sizeof(sb2_geo_cell)) || b.ndim != 1)
        throw std::runtime_error("geo cells: a 1-d array of 96-byte geo_cell_data records is required (shyft_b200.geo_cell_data_vector)");
    std::vector<sb::geo_cell_data> v(size_t(b.shape[0]));
    if (b.strides[0] != b.itemsize) throw std::runtime_error("geo cells: the record array must be contiguous");
    std::memcpy(v.data(), b.ptr, v.size() * sizeof(sb2_geo_cell));
    return v;
}

sb::region_environment env_from(const py::dict& d) {
    sb::region_environment env;
    auto take = [&](const char* name, sb::geo_point_sources& s) {
        if (!d.contains(name)) return;
        const py::tuple t = d[name].cast<py::tuple>();
        s.xyz = flat(t[0].cast<darray>());
        s.values = flat(t[1].cast<darray>());
    };
    take("temperature", env.temperature); take("precipitation", env.precipitation); take("radiation", env.radiation);
    take("wind_speed", env.wind_speed); take("rel_hum", env.rel_hum);
    return env;
}

template <int STACK>
std::unique_ptr<sb::region_model<STACK>> make_model(const py::array& geo, const std::vector<double>& region_parameter, int device, int collect_bits) {
    auto p = std::make_unique<sb::region_model<STACK>>(geo_vector(geo), region_parameter, device);
    p->set_collector_mode(collect_bits);
    return p;
}

template <int STACK>
void bind_model(py::module_& m, const char* name, int collect_bits, const char* doc) {
    using M = sb::region_model<STACK>;
    py::class_<M>(m, name, doc)
        .def(py::init([collect_bits](const py::array& geo, const std::vector<double>& region_parameter, int device) {
                 return make_model<STACK>(geo, region_parameter, device, collect_bits);
             }),
             py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0)
        .def("size", &M::size)
        .def("number_of_catchments", &M::number_of_catchments)
        .def_property_readonly("catchment_ids", &M::catchment_ids)
        .def("set_region_parameter", &M::set_region_parameter, py::arg("p"))
        .def("get_region_parameter", &M::get_region_parameter)
        .def("set_catchment_parameter", &M::set_catchment_parameter, py::arg("catchment_id"), py::arg("p"))
        .def("remove_catchment_parameter", &M::remove_catchment_parameter, py::arg("catchment_id"))
        .def("has_catchment_parameter", &M::has_catchment_parameter, py::arg("catchment_id"))
        .def("get_catchment_parameter", &M::get_catchment_parameter, py::arg("catchment_id"))
        .def("set_catchment_calculation_filter", &M::set_catchment_calculation_filter, py::arg("catchment_id_list"))
        .def("set_states", [](M& self, const darray& states) { self.set_states(flat(states)); }, py::arg("states"))
        .def("get_states",
             [](const M& self) {
                 std::vector<double> s;
                 self.get_states(s);
                 const py::ssize_t n = py::ssize_t(self.size());
                 darray out({n, n ? py::ssize_t(s.size()) / n : py::ssize_t(0)});
                 std::memcpy(out.mutable_data(), s.data(), s.size() * sizeof(double));
                 return out;
             })
        .def("revert_to_initial_state", &M::revert_to_initial_state)
        .def("adjust_q", &M::adjust_q, py::arg("q_scale"), py::arg("cids"))
        .def("adjust_state_to_target_flow", &M::adjust_state_to_target_flow, py::arg("wanted_flow_m3s"), py::arg("cids"), py::arg("start_step") = 0,
             py::arg("scale_range") = 3.0, py::arg("scale_eps") = 1.0e-3, py::arg("max_iter") = 300, py::arg("n_steps") = 1)
        .def("initialize_cell_environment",
             [](M& self, int64_t t0_us, int64_t dt_us, size_t n) { self.initialize_cell_environment(sb::fixed_dt{t0_us, dt_us, n}); },
             py::arg("t0_us"), py::arg("dt_us"), py::arg("n"))
        .def("interpolate",
             [](M& self, const py::dict& env, bool best_effort) { return self.interpolate(self.ip_parameter, env_from(env), best_effort); },
             py::arg("env"), py::arg("best_effort") = true)
        .def("run_interpolation",
             [](M& self, int64_t t0_us, int64_t dt_us, size_t n, const py::dict& env, bool best_effort) {
                 return self.run_interpolation(self.ip_parameter, sb::fixed_dt{t0_us, dt_us, n}, env_from(env), best_effort);
             },
             py::arg("t0_us"), py::arg("dt_us"), py::arg("n"), py::arg("env"), py::arg("best_effort") = true,
             "run_interpolation(interpolation_parameter defaults, fixed_dt{t0, dt, n} in microseconds, {name: (xyz [s][3], values [n][s])})")
        .def("is_cell_env_ts_ok", &M::is_cell_env_ts_ok)
        .def("run_cells", &M::run_cells, py::arg("use_ncore") = 0, py::arg("start_step") = 0, py::arg("n_steps") = 0)
        .def("run_ensemble",
             [](M& self, const py::list& members, int start_step, int n_steps, int window_steps) {
                 std::vector<sb::region_environment> envs;
                 for (const py::handle& d : members) envs.push_back(env_from(d.cast<py::dict>()));
                 const auto r = self.run_ensemble(self.ip_parameter, envs, start_step, n_steps, window_steps);
                 auto to_array = [](const std::vector<std::vector<std::vector<double>>>& v) {
                     const py::ssize_t E = py::ssize_t(v.size()), K = E ? py::ssize_t(v[0].size()) : 0, T = K ? py::ssize_t(v[0][0].size()) : 0;
                     darray out({E, K, T});
                     for (py::ssize_t e = 0; e < E; ++e)
                         for (py::ssize_t k = 0; k < K; ++k) std::memcpy(out.mutable_data(e, k, 0), v[size_t(e)][size_t(k)].data(), size_t(T) * sizeof(double));
                     return out;
                 };
                 return py::make_tuple(to_array(r.discharge), to_array(r.charge));
             },
             py::arg("members"), py::arg("start_step") = 0, py::arg("n_steps") = 0, py::arg("window_steps") = 4096,
             "forcing ensemble: a list of run_interpolation's dicts, one per member -> (discharge, charge), each [member][catchment][step]")
        .def("catchment_discharges",
             [](const M& self) {
                 std::vector<std::vector<double>> cr;
                 self.catchment_discharges(cr);
                 darray out({py::ssize_t(cr.size()), py::ssize_t(cr.empty() ? 0 : cr[0].size())});
                 for (size_t k = 0; k < cr.size(); ++k) std::memcpy(out.mutable_data(py::ssize_t(k), 0), cr[k].data(), cr[k].size() * sizeof(double));
                 return out;
             },
             "[catchment][step], the TSV of region_model::catchment_discharges (core/region_model.h:873-885)")
        .def("response",
             [](const M& self, int series) {
                 const std::vector<double> v = self.response(series);
                 darray out({py::ssize_t(self.time_axis.n), py::ssize_t(self.size())});
                 std::memcpy(out.mutable_data(), v.data(), v.size() * sizeof(double));
                 return out;
             },
             py::arg("series"))
        .def("set_river_network",
             [](M& self, const darray& rivers) { self.set_river_network(flat(rivers)); }, py::arg("rivers"),
             "rivers [n][6] = id, downstream id, downstream distance, uhg velocity, alpha, beta (core/routing.h:98-123)")
        .def("river_output_flow_m3s", &M::river_output_flow_m3s, py::arg("river_id"))
        .def("statistics", &M::statistics, py::arg("kind"), py::arg("series"), py::arg("indexes"), py::arg("op"), py::arg("scope") = int(SB2_SCOPE_CATCHMENT_IX))
        .def("statistics_value", &M::statistics_value, py::arg("kind"), py::arg("series"), py::arg("indexes"), py::arg("ith_timestep"), py::arg("op"),
             py::arg("scope") = int(SB2_SCOPE_CATCHMENT_IX));
}

// model_calibrator<RegionModel>(optimizer_name) of api/boostpython/expose.h:472-731: the optimizer class of one model type under the
// reference's member names.  keep_alive ties the model's lifetime to the optimizer that holds a reference to it.
template <int STACK>
void bind_optimizer(py::module_& m, const char* name) {
    using O = sb::optimizer<STACK>;
    using M = sb::region_model<STACK>;
    using P = std::vector<double>;
    py::class_<O>(m, name, "optimizer<region_model, parameter, ts> (core/model_calibration.h:404-900): goal-function entry on the device, search drivers on the host")
        .def(py::init<M&, const std::vector<sb::target_specification>&, const P&, const P&>(), py::arg("model"), py::arg("targets"), py::arg("p_min"),
             py::arg("p_max"), py::keep_alive<1, 2>())
        .def(py::init<M&>(), py::arg("model"), py::keep_alive<1, 2>())
        .def("set_target_specification", &O::set_target_specification, py::arg("target_specification"), py::arg("parameter_lower_bound"),
             py::arg("parameter_upper_bound"))
        .def("set_parameter_ranges", &O::set_parameter_ranges, py::arg("p_min"), py::arg("p_max"))
        .def("set_verbose_level", &O::set_verbose_level, py::arg("level"))
        .def("reset_states", &O::reset_states)
        .def("calculate_goal_function", &O::calculate_goal_function, py::arg("full_vector_of_parameters"))
        .def("calculate_goal_function_batch",
             [](O& self, const darray& P) {
                 if (P.ndim() != 2) throw std::runtime_error("calculate_goal_function_batch: parameters must be [n_sets][parameter_size]");
                 std::vector<std::vector<double>> sets(size_t(P.shape(0)), std::vector<double>(size_t(P.shape(1))));
                 for (py::ssize_t k = 0; k < P.shape(0); ++k) std::memcpy(sets[size_t(k)].data(), P.data(k, 0), size_t(P.shape(1)) * sizeof(double));
                 return self.calculate_goal_function_batch(sets);
             },
             py::arg("parameter_sets"), "a whole population in one device pass; equals calling calculate_goal_function once per set")
        .def("optimize", &O::optimize, py::arg("p"), py::arg("max_n_evaluations"), py::arg("tr_start"), py::arg("tr_stop"))
        .def("optimize_dream", &O::optimize_dream, py::arg("p"), py::arg("max_n_evaluations"))
        .def("optimize_sceua", &O::optimize_sceua, py::arg("p"), py::arg("max_n_evaluations"), py::arg("x_eps"), py::arg("y_eps"))
        .def("parameter_active", &O::active_parameter, py::arg("i"))
        .def_property_readonly("trace_size", &O::trace_size)
        .def_readonly("trace_goal_function_values", &O::goal_fn_trace)
        .def("trace_goal_function_value", &O::trace_goal_function_value, py::arg("i"))
        .def("trace_parameter", &O::trace_parameter, py::arg("i"))
        .def_readonly("target_specification", &O::targets)
        .def_readonly("parameter_lower_bound", &O::parameter_lower_bound)
        .def_readonly("parameter_upper_bound", &O::parameter_upper_bound)
        .def_readonly("n_single_calls", &O::n_single_calls)
        .def_readonly("n_batch_calls", &O::n_batch_calls);
}

}  // namespace

PYBIND11_MODULE(_shyft_b200_cpp, m) {
    m.doc() = "pybind11 binding of shyft_b200's C++ region-model shim (names of api/boostpython/expose.h)";
    py::class_<sb::q_adjust_result>(m, "FlowAdjustResult", "q_adjust_result (core/model_state_tuning.h:11-16)")
        .def_readonly("q_0", &sb::q_adjust_result::q_0)
        .def_readonly("q_r", &sb::q_adjust_result::q_r)
        .def_readonly("diagnostics", &sb::q_adjust_result::diagnostics);
    const int all = SB2_COLLECT_ALL, opt = SB2_COLLECT_DISCHARGE;
    bind_model<SB2_PT_GS_K>(m, "PTGSKModel", all, "region_model<pt_gs_k::cell_complete_response_t> (api/boostpython/expose.h, shyft/api/pt_gs_k)");
    bind_model<SB2_PT_HS_K>(m, "PTHSKModel", all, "region_model<pt_hs_k::cell_complete_response_t>");
    bind_model<SB2_HBV_STACK>(m, "HbvModel", all, "region_model<hbv_stack::cell_complete_response_t>");
    bind_model<SB2_PT_SS_K>(m, "PTSSKModel", all, "region_model<pt_ss_k::cell_complete_response_t>");
    bind_model<SB2_PT_HPS_K>(m, "PTHPSKModel", all, "region_model<pt_hps_k::cell_complete_response_t>");
    // the *OptModel types are the same C++ classes with the discharge collector only (cell_discharge_response_t): factory functions
    m.def("PTGSKOptModel", [opt](const py::array& geo, const std::vector<double>& p, int device) { return make_model<SB2_PT_GS_K>(geo, p, device, opt); },
          py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0);
    m.def("PTHSKOptModel", [opt](const py::array& geo, const std::vector<double>& p, int device) { return make_model<SB2_PT_HS_K>(geo, p, device, opt); },
          py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0);
    m.def("PTSSKOptModel", [opt](const py::array& geo, const std::vector<double>& p, int device) { return make_model<SB2_PT_SS_K>(geo, p, device, opt); },
          py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0);
    m.def("PTHPSKOptModel", [opt](const py::array& geo, const std::vector<double>& p, int device) { return make_model<SB2_PT_HPS_K>(geo, p, device, opt); },
          py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0);
    m.def("HbvOptModel", [opt](const py::array& geo, const std::vector<double>& p, int device) { return make_model<SB2_HBV_STACK>(geo, p, device, opt); },
          py::arg("geo_cell_data_vector"), py::arg("region_parameter"), py::arg("device") = 0);
    // TargetSpecificationPts / TargetSpecificationVector (api/boostpython/api_target_specification.cpp:50-61); the vector is a Python list
    py::class_<sb::target_specification>(m, "TargetSpecificationPts", "target_specification<pts_t> (core/model_calibration.h:242-329)")
        .def(py::init([](const std::vector<double>& values, int64_t t0_us, int64_t dt_us, const std::vector<int64_t>& cids, double scale_factor, int calc_mode,
                         double s_r, double s_a, double s_b, int catchment_property, int64_t river_id, const std::string& uid,
                         const std::vector<int64_t>& period_points_us) {
                 sb::target_specification t;
                 t.values = values; t.t0_us = t0_us; t.dt_us = dt_us; t.catchment_indexes = cids; t.scale_factor = scale_factor; t.calc_mode = calc_mode;
                 t.s_r = s_r; t.s_a = s_a; t.s_b = s_b; t.catchment_property = catchment_property; t.river_id = river_id; t.uid = uid;
                 t.period_points_us = period_points_us;
                 return t;
             }),
             py::arg("values"), py::arg("t0_us"), py::arg("dt_us"), py::arg("catchment_indexes") = std::vector<int64_t>{}, py::arg("scale_factor") = 1.0,
             py::arg("calc_mode") = int(sb::NASH_SUTCLIFFE), py::arg("s_r") = 1.0, py::arg("s_a") = 1.0, py::arg("s_b") = 1.0,
             py::arg("catchment_property") = int(sb::DISCHARGE), py::arg("river_id") = 0, py::arg("uid") = std::string(),
             py::arg("period_points_us") = std::vector<int64_t>{})
        .def_readwrite("values", &sb::target_specification::values)
        .def_readwrite("catchment_indexes", &sb::target_specification::catchment_indexes)
        .def_readwrite("scale_factor", &sb::target_specification::scale_factor)
        .def_readwrite("calc_mode", &sb::target_specification::calc_mode)
        .def_readwrite("catchment_property", &sb::target_specification::catchment_property)
        .def_readwrite("s_r", &sb::target_specification::s_r)
        .def_readwrite("s_a", &sb::target_specification::s_a)
        .def_readwrite("s_b", &sb::target_specification::s_b)
        .def_readwrite("river_id", &sb::target_specification::river_id)
        .def_readwrite("uid", &sb::target_specification::uid)
        .def_readwrite("period_points_us", &sb::target_specification::period_points_us);
    m.def("calendar_period_points",
          [](int64_t t0_us, const std::string& unit, size_t n) {
              const sb::calendar_unit u = unit == "day" ? sb::CAL_DAY : unit == "week" ? sb::CAL_WEEK : unit == "month" ? sb::CAL_MONTH
                                          : unit == "quarter" ? sb::CAL_QUARTER : unit == "year" ? sb::CAL_YEAR : sb::calendar_unit(-1);
              if (int(u) < 0) throw std::runtime_error("calendar_period_points: unit must be day, week, month, quarter or year");
              return sb::calendar_period_points(t0_us, u, n);
          },
          py::arg("t0_us"), py::arg("unit"), py::arg("n"),
          "n + 1 boundaries of n calendar periods from t0 (UTC): a calendar_dt target axis as the point axis period_points_us takes");
    bind_optimizer<SB2_PT_GS_K>(m, "PTGSKOptimizer");
    bind_optimizer<SB2_PT_HS_K>(m, "PTHSKOptimizer");
    bind_optimizer<SB2_HBV_STACK>(m, "HbvOptimizer");
    bind_optimizer<SB2_PT_SS_K>(m, "PTSSKOptimizer");
    bind_optimizer<SB2_PT_HPS_K>(m, "PTHPSKOptimizer");
    m.attr("NASH_SUTCLIFFE") = int(sb::NASH_SUTCLIFFE); m.attr("KLING_GUPTA") = int(sb::KLING_GUPTA); m.attr("ABS_DIFF") = int(sb::ABS_DIFF);
    m.attr("RMSE") = int(sb::RMSE); m.attr("DISCHARGE") = int(sb::DISCHARGE); m.attr("SNOW_COVERED_AREA") = int(sb::SNOW_COVERED_AREA);
    m.attr("SNOW_WATER_EQUIVALENT") = int(sb::SNOW_WATER_EQUIVALENT); m.attr("ROUTED_DISCHARGE") = int(sb::ROUTED_DISCHARGE);
    m.attr("CELL_CHARGE") = int(sb::CELL_CHARGE);
    m.attr("STAT_FORCING") = int(SB2_STAT_FORCING); m.attr("STAT_RESPONSE") = int(SB2_STAT_RESPONSE); m.attr("STAT_STATE") = int(SB2_STAT_STATE);
    m.attr("STAT_SUM") = int(SB2_STAT_SUM); m.attr("STAT_AREA_AVERAGE") = int(SB2_STAT_AREA_AVERAGE);
    m.attr("R_AVG_DISCHARGE") = int(SB2_R_AVG_DISCHARGE); m.attr("R_CHARGE_M3S") = int(SB2_R_CHARGE_M3S);
}
