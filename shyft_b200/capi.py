"""ctypes binding of the C ABI in include/shyft_b200.h (shyft_b200/libshyft_b200.so).

There is no CPU fallback: loading fails loudly when the CUDA library is missing, and model creation
fails loudly when no CUDA device is present.
"""
import ctypes as C
import os

import numpy as np

from . import _build

c_dp = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)

# enums of include/shyft_b200.h
PT_GS_K, PT_HS_K, HBV_STACK, PT_SS_K, PT_HPS_K = 0, 1, 2, 3, 4
TEMPERATURE, PRECIPITATION, RADIATION, WIND_SPEED, REL_HUM = 0, 1, 2, 3, 4
FORCING_NAMES = ("temperature", "precipitation", "radiation", "wind_speed", "rel_hum")
TIME_MAJOR, CELL_MAJOR = 0, 1
COLLECT_NONE, COLLECT_DISCHARGE, COLLECT_SNOW, COLLECT_ALL, COLLECT_STATE = 0, 1, 2, 7, 8
RESPONSE_NAMES = ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output", "soil_outflow")
STATE_SERIES_NAMES = {
    PT_GS_K: ("kirchner_discharge", "gs_albedo", "gs_lwc", "gs_surface_heat", "gs_alpha", "gs_sdc_melt_mean", "gs_acc_melt", "gs_iso_pot_energy",
              "gs_temp_swe"),
    PT_HS_K: ("kirchner_discharge", "snow_sca", "snow_swe") + tuple(f"snow_sp_{i}" for i in range(5)) + tuple(f"snow_sw_{i}" for i in range(5)),
    PT_SS_K: ("kirchner_discharge", "snow_swe", "snow_sca", "snow_alpha", "snow_nu", "snow_lwc", "snow_residual"),
    PT_HPS_K: ("kirchner_discharge", "snow_sca", "snow_swe", "snow_surface_heat") + tuple(f"snow_sp_{i}" for i in range(5))
    + tuple(f"snow_sw_{i}" for i in range(5)) + tuple(f"snow_albedo_{i}" for i in range(5)) + tuple(f"snow_iso_pot_energy_{i}" for i in range(5)),
    HBV_STACK: ("snow_swe", "snow_sca", "soil_moisture", "tank_uz", "tank_lz") + tuple(f"snow_sp_{i}" for i in range(5))
    + tuple(f"snow_sw_{i}" for i in range(5)),
}

# sb2_geo_cell, 12 x 8 bytes, no padding
GEO_DTYPE = np.dtype([("x", "f8"), ("y", "f8"), ("z", "f8"), ("area", "f8"), ("catchment_id", "i8"), ("radiation_slope_factor", "f8"),
                      ("glacier", "f8"), ("lake", "f8"), ("reservoir", "f8"), ("forest", "f8"), ("routing_id", "i8"), ("routing_distance", "f8")])


class IdwParameter(C.Structure):
    _fields_ = [("max_members", C.c_int64), ("max_distance", C.c_double), ("distance_measure_factor", C.c_double), ("zscale", C.c_double),
                ("default_temp_gradient", C.c_double), ("gradient_by_equation", C.c_int32), ("scale_factor", C.c_double)]


class BtkParameter(C.Structure):
    _fields_ = [("gradient_sd", C.c_double), ("sill", C.c_double), ("nug", C.c_double), ("range", C.c_double), ("zscale", C.c_double)]


class InterpolationParameter(C.Structure):
    """interpolation_parameter (core/region_model.h:65-95); default-constructed values via the library."""
    _fields_ = [("temperature", BtkParameter), ("use_idw_for_temperature", C.c_int32), ("temperature_idw", IdwParameter),
                ("precipitation", IdwParameter), ("wind_speed", IdwParameter), ("radiation", IdwParameter), ("rel_hum", IdwParameter)]

    def __init__(self, **kw):
        super().__init__()
        lib().sb2_interpolation_parameter_default(C.byref(self))
        for k, v in kw.items():
            setattr(self, k, v)


class Target(C.Structure):
    """sb2_target: target_specification (core/model_calibration.h:242-329)"""
    _fields_ = [("values", c_dp), ("t0_us", C.c_int64), ("dt_us", C.c_int64), ("n", C.c_int64), ("catchment_ids", c_i64p),
                ("n_catchments", C.c_int32), ("river_id", C.c_int64), ("scale_factor", C.c_double), ("calc_mode", C.c_int32),
                ("property", C.c_int32), ("s_r", C.c_double), ("s_a", C.c_double), ("s_b", C.c_double), ("period_points_us", c_i64p)]


class QAdjustResult(C.Structure):
    """sb2_q_adjust_result: q_adjust_result (core/model_state_tuning.h:11-16)"""
    _fields_ = [("q_0", C.c_double), ("q_r", C.c_double), ("_diagnostics", C.c_char * 512)]

    @property
    def diagnostics(self):
        return self._diagnostics.decode()


EXPORTS = """sb2_interpolation_parameter_default sb2_model_create sb2_model_destroy sb2_last_error sb2_version sb2_size
sb2_number_of_catchments sb2_catchment_ids sb2_cell_catchment_ix sb2_parameter_size sb2_state_size sb2_set_region_parameter
sb2_get_region_parameter sb2_set_catchment_parameter sb2_get_catchment_parameter sb2_remove_catchment_parameter
sb2_has_catchment_parameter sb2_set_catchment_calculation_filter sb2_set_states sb2_get_states sb2_set_initial_state
sb2_hbv_distribute_snow sb2_get_initial_state sb2_revert_to_initial_state sb2_adjust_q sb2_adjust_state_to_target_flow sb2_extract_state sb2_apply_state sb2_set_collector_mode sb2_initialize_cell_environment
sb2_set_cell_forcing sb2_get_cell_forcing sb2_set_sources sb2_set_sources_on_axis sb2_set_sources_on_axes sb2_get_sources_on_model_axis sb2_interpolate sb2_is_cell_env_ts_ok sb2_run_cells sb2_run_windowed
sb2_set_ensemble_sources sb2_set_ensemble_sources_on_axis sb2_run_ensemble
sb2_get_response sb2_get_state_series sb2_catchment_discharges sb2_catchment_charges sb2_statistics_series sb2_statistics_cells
sb2_statistics_geo sb2_set_river_network sb2_river_flows
sb2_set_targets sb2_calculate_goal_function sb2_calculate_goal_function_batch sb2_unit_eval sb2_host_eval sb2_set_idw_dense sb2_set_stream sb2_device_catchment_discharges sb2_device_catchment_charges sb2_step_chunk_steps sb2_check_guards sb2_kernel_launches sb2_last_run_kernel_ms""".split()

_LIB = None


def library_path():
    return _build.LIB


def lib():
    """Load (building if stale and nvcc is present) the CUDA library.  Raises if it cannot be had."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("SB2_LIB") or _build.LIB   # SB2_LIB: another build of the library, e.g. for an A/B timing
    if not os.path.exists(path) or os.environ.get("SB2_REBUILD"):
        try:  # normally __graft_entry__.build() has produced the file and it travels with the tree
            _build.build_library(force=bool(os.environ.get("SB2_REBUILD")))
        except Exception as e:
            raise RuntimeError(f"shyft_b200: CUDA library {path} is missing and could not be built ({e}); there is no CPU fallback") from e
    L = C.CDLL(path)
    L.sb2_last_error.restype = C.c_char_p
    L.sb2_last_error.argtypes = [C.c_void_p]
    for name in ("sb2_size", "sb2_number_of_catchments", "sb2_kernel_launches"):
        getattr(L, name).restype = C.c_int64
        getattr(L, name).argtypes = [C.c_void_p]
    L.sb2_model_destroy.restype = None
    L.sb2_model_destroy.argtypes = [C.c_void_p]
    L.sb2_interpolation_parameter_default.restype = None
    _LIB = L
    return L


def dptr(a):
    return a.ctypes.data_as(c_dp) if a is not None else None


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


UNIT_FUNCTIONS = dict(exp=(0, 1, 1), log=(1, 1, 1), pow=(2, 2, 1), lgamma=(3, 1, 1), gamma_p=(4, 2, 1), corr_lwc=(5, 5, 1), calc_snow_state=(6, 7, 2),
                      kirchner_step=(7, 7, 3),
                      # the forms the production kernels use (sb2_unit.cuh)
                      exp_flat=(8, 1, 1), log_flat=(9, 1, 1), pow_flat=(10, 2, 1), kirchner_step_warp=(11, 7, 3),
                      div_by=(12, 2, 2), kirchner_step_warp_udt=(13, 7, 3), skaugen_step=(14, 18, 11), sca_rel_red=(15, 4, 2),
                      hps_step=(16, 41, 27))


def check_guards():
    """-> (violations, first finding): the red zones of every live device buffer (SB2_GUARD=1), see sb2_check_guards"""
    buf = C.create_string_buffer(256)
    L = lib()
    L.sb2_check_guards.restype = C.c_int64
    return int(L.sb2_check_guards(buf, C.c_int(256))), buf.value.decode()


def host_eval(fn, inputs, n_out):
    """sb2_host_eval: a host-side algorithm of the library (no device needed) -> out [n_out]"""
    a = f64(inputs).ravel()
    out = np.zeros(n_out)
    if lib().sb2_host_eval(C.c_int(fn), dptr(a), C.c_int(a.size), dptr(out), C.c_int(n_out)) != 0:
        raise RuntimeError("sb2_host_eval: bad arguments")
    return out


def unit_eval(fn, inputs, device=0):
    """Evaluate one device function row-wise: inputs [n][n_in] -> [n][n_out] (sb2_unit_eval)."""
    code, n_in, n_out = UNIT_FUNCTIONS[fn]
    a = f64(inputs).reshape(-1, n_in)
    out = np.zeros((a.shape[0], n_out))
    rc = lib().sb2_unit_eval(C.c_int(device), C.c_int(code), C.c_int64(a.shape[0]), dptr(a), C.c_int(n_in), dptr(out), C.c_int(n_out))
    if rc != 0:
        raise RuntimeError(lib().sb2_last_error(None).decode())
    return out
