"""Python mirror of the reference's region-model surface over the C ABI.

Names, argument meaning and error behaviour follow region_model<cell_t> (core/region_model.h:211-1049) as exposed to
Python by api/boostpython/expose.h:143-430 (`PTGSKModel`, `PTGSKOptModel`, ...): `run_interpolation`, `interpolate`,
`run_cells`, `get_states` / `set_states` / `revert_to_initial_state`, `set_region_parameter` / `set_catchment_parameter`,
`set_catchment_calculation_filter`, `catchment_discharges`, river flow accessors.  Errors that are `std::runtime_error`
in the reference surface as `RuntimeError` with the same message.  All numerics run in the CUDA library; this module only
moves numpy arrays across the ABI.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import (COLLECT_ALL, COLLECT_DISCHARGE, COLLECT_NONE, COLLECT_SNOW, COLLECT_STATE, FORCING_NAMES, GEO_DTYPE, HBV_STACK, PT_GS_K, PT_HPS_K, PT_HS_K, PT_SS_K,
                   RESPONSE_NAMES, STATE_SERIES_NAMES, InterpolationParameter, dptr, f64)

# parameter vector names, order of parameter::get_name (core/pt_gs_k.h:156-193, core/pt_hs_k.h:133-146, core/hbv_stack.h:136-167)
PARAMETER_NAMES = {
    PT_GS_K: ("kirchner.c1", "kirchner.c2", "kirchner.c3", "ae.ae_scale_factor", "gs.tx", "gs.wind_scale", "gs.max_water", "gs.wind_const",
              "gs.fast_albedo_decay_rate", "gs.slow_albedo_decay_rate", "gs.surface_magnitude", "gs.max_albedo", "gs.min_albedo",
              "gs.snowfall_reset_depth", "gs.snow_cv", "gs.glacier_albedo", "p_corr.scale_factor", "gs.snow_cv_forest_factor",
              "gs.snow_cv_altitude_factor", "pt.albedo", "pt.alpha", "gs.initial_bare_ground_fraction", "gs.winter_end_day_of_year",
              "gs.calculate_iso_pot_energy", "gm.dtf", "routing.velocity", "routing.alpha", "routing.beta", "gs.n_winter_days",
              "gm.direct_response", "msp.reservoir_direct_response_fraction"),
    PT_HS_K: ("kirchner.c1", "kirchner.c2", "kirchner.c3", "ae.ae_scale_factor", "hs.lw", "hs.tx", "hs.cx", "hs.ts", "hs.cfr", "gm.dtf",
              "p_corr.scale_factor", "pt.albedo", "pt.alpha", "routing.velocity", "routing.alpha", "routing.beta", "gm.direct_response",
              "msp.reservoir_direct_response_fraction"),
    PT_SS_K: ("kirchner.c1", "kirchner.c2", "kirchner.c3", "ae.ae_scale_factor", "ss.alpha_0", "ss.d_range", "ss.unit_size", "ss.max_water_fraction",
              "ss.tx", "ss.cx", "ss.ts", "ss.cfr", "p_corr.scale_factor", "pt.albedo", "pt.alpha", "gm.dtf", "routing.velocity", "routing.alpha",
              "routing.beta", "gm.direct_response", "msp.reservoir_direct_response_fraction"),
    PT_HPS_K: ("kirchner.c1", "kirchner.c2", "kirchner.c3", "ae.ae_scale_factor", "hps.lw", "hps.tx", "hps.cfr", "hps.wind_scale", "hps.wind_const",
               "hps.surface_magnitude", "hps.max_albedo", "hps.min_albedo", "hps.fast_albedo_decay_rate", "hps.slow_albedo_decay_rate",
               "hps.snowfall_reset_depth", "hps.calculate_iso_pot_energy", "gm.dtf", "p_corr.scale_factor", "pt.albedo", "pt.alpha",
               "routing.velocity", "routing.alpha", "routing.beta", "msp.reservoir_direct_response_fraction"),
    HBV_STACK: ("soil.fc", "soil.beta", "ae.lp", "tank.uz1", "tank.kuz2", "tank.kuz1", "tank.perc", "tank.klz", "hs.lw", "hs.tx", "hs.cx", "hs.ts",
                "hs.cfr", "p_corr.scale_factor", "pt.albedo", "pt.alpha", "gm.dtf", "routing.velocity", "routing.alpha", "routing.beta",
                "gm.direct_response", "msp.reservoir_direct_response_fraction"),
}
USEC = 1000000


def geo_cell_data_vector(x, y, z, area=1.0e6, catchment_id=1, radiation_slope_factor=0.9, glacier=0.0, lake=0.0, reservoir=0.0, forest=0.0,
                         routing_id=0, routing_distance=0.0):
    """Structure-of-arrays constructor for a vector of geo_cell_data (core/geo_cell_data.h:107-138) -> numpy record array."""
    n = np.size(x)
    g = np.zeros(n, dtype=GEO_DTYPE)
    for name, v in (("x", x), ("y", y), ("z", z), ("area", area), ("catchment_id", catchment_id),
                    ("radiation_slope_factor", radiation_slope_factor), ("glacier", glacier), ("lake", lake), ("reservoir", reservoir),
                    ("forest", forest), ("routing_id", routing_id), ("routing_distance", routing_distance)):
        g[name] = v
    return g


class TimeAxis:
    """time_axis::fixed_dt (core/time_axis.h:74-115); start and delta in whole seconds like the reference's Python API."""

    def __init__(self, start, delta_t, n):
        self.start, self.delta_t, self.n = int(start), int(delta_t), int(n)

    def size(self):
        return self.n

    def time(self, i):
        return self.start + i * self.delta_t


class GeoPointSources:
    """The geo-located series of one variable on their OWN point axis (vector<geo_point_ts>, api/api.h:137-168): `times` [P] point
    times in seconds (strictly increasing, shared by the S series), `t_end` the series' total_period().end in seconds, `values`
    [P][S], `point_fx` "average" (stair-case, POINT_AVERAGE_VALUE) or "instant" (linear between points).  The projection onto the
    model axis (average_accessor, core/time_series.h:202-310, 2033-2072) runs on the device when the environment is set."""

    def __init__(self, xyz, times, values, t_end=None, point_fx="average"):
        self.xyz, self.values = f64(xyz), f64(values)
        self.times_us = np.ascontiguousarray(np.round(np.asarray(times, dtype=np.float64) * USEC), dtype=np.int64)
        if t_end is None:  # a fixed-interval series ends one interval after its last point
            t_end = times[-1] + (times[-1] - times[-2]) if len(times) > 1 else times[-1]
        self.t_end_us = int(round(float(t_end) * USEC))
        if point_fx not in ("average", "instant"):
            raise RuntimeError("point_fx must be 'average' or 'instant'")
        self.point_fx = point_fx


class GeoPointSourceVector:
    """vector<geo_point_ts> whose series each have their own point axis: a list of (xyz, times [s], values, t_end [s] or None, point_fx)
    -- one entry per station (api/api.h:137-168)."""

    def __init__(self, sources):
        xyz, n_points, t, v, t_end, fx = [], [], [], [], [], []
        for x, times, values, end, point_fx in sources:
            times = np.asarray(times, dtype=np.float64)
            values = f64(values).ravel()
            if values.size != times.size:
                raise RuntimeError("a source needs one value per point")
            if point_fx not in ("average", "instant"):
                raise RuntimeError("point_fx must be 'average' or 'instant'")
            if end is None:
                end = times[-1] + (times[-1] - times[-2]) if times.size > 1 else times[-1]
            xyz.append(x); n_points.append(times.size); t.append(np.round(times * USEC).astype(np.int64)); v.append(values)
            t_end.append(int(round(float(end) * USEC))); fx.append(1 if point_fx == "instant" else 0)
        self.xyz = f64(xyz).reshape(-1, 3)
        self.n_points = np.ascontiguousarray(n_points, dtype=np.int64)
        self.times_us = np.ascontiguousarray(np.concatenate(t) if t else np.zeros(0), dtype=np.int64)
        self.values = f64(np.concatenate(v) if v else np.zeros(0))
        self.t_end_us = np.ascontiguousarray(t_end, dtype=np.int64)
        self.point_fx = np.ascontiguousarray(fx, dtype=np.int32)


class RegionEnvironment:
    """a_region_environment (api/api.h:137-168): per variable a set of geo-located series.

    `env.temperature = (xyz [S,3], values [T,S])` for series already on the model axis, or a `GeoPointSources` for series on their
    own axis (3-hourly, daily, irregular ...); a variable left as None keeps the cells' series NaN (region_model.h:448-452).
    """

    def __init__(self, **kw):
        for name in FORCING_NAMES:
            setattr(self, name, kw.get(name))


def _stats():
    from . import statistics
    return statistics


class RegionModel:
    stack = PT_GS_K
    default_collect = COLLECT_ALL | COLLECT_STATE  # the "complete response" cell type (pt_gs_k_cell_model.h:210)

    def __init__(self, geo_cells, region_parameter=None, device=0):
        self._L = capi.lib()
        geo = np.ascontiguousarray(geo_cells, dtype=GEO_DTYPE)
        self._h = C.c_void_p()
        rc = self._L.sb2_model_create(C.c_int(self.stack), C.c_int64(geo.shape[0]), geo.ctypes.data_as(C.c_void_p), C.c_int(device),
                                      C.byref(self._h))
        if rc != 0:
            raise RuntimeError(self._L.sb2_last_error(None).decode())
        self.geo = geo
        self.time_axis = None
        self.ip_parameter = None
        self.region_env = None
        self._collect = self.default_collect
        self._state_collection = False
        self._snow_collection = False
        self._apply_collect()
        if region_parameter is not None:
            self.set_region_parameter(region_parameter)

    # -- plumbing -------------------------------------------------------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(self._L.sb2_last_error(self._h).decode())

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                self._L.sb2_model_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    def _apply_collect(self):
        bits = self._collect
        if self.default_collect & COLLECT_STATE:  # complete-response cells: state series only when switched on (:844-849)
            bits = (bits & ~COLLECT_STATE) | (COLLECT_STATE if self._state_collection else 0)
        else:                                     # discharge-collector cells: optional sca/swe (:851-858)
            bits = (bits & ~COLLECT_SNOW) | (COLLECT_SNOW if self._snow_collection else 0)
        self._ck(self._L.sb2_set_collector_mode(self._h, C.c_int(bits)))
        self._bits = bits

    # -- sizes / indexing --------------------------------------------------------------------------------------------
    @property
    def statistics(self):
        """basic_cell_statistics over this model's cells (model.statistics.discharge(cids), .temperature(cids), ...; api/api.h:179-420)"""
        return _stats().BasicCellStatistics(self)

    @property
    def state(self):
        """state_io_handler of this model's cells (model.state.extract_state(cids) / .apply_state(states, cids); api/api_state.h:93-142)"""
        from .state_io import StateIoHandler
        return StateIoHandler(self)

    def size(self):
        return int(self._L.sb2_size(self._h))

    def number_of_catchments(self):
        return int(self._L.sb2_number_of_catchments(self._h))

    @property
    def catchment_ids(self):
        out = np.zeros(self.number_of_catchments(), dtype=np.int64)
        self._ck(self._L.sb2_catchment_ids(self._h, out.ctypes.data_as(capi.c_i64p)))
        return out

    def cell_catchment_ix(self):
        out = np.zeros(self.size(), dtype=np.int64)
        self._ck(self._L.sb2_cell_catchment_ix(self._h, out.ctypes.data_as(capi.c_i64p)))
        return out

    @property
    def parameter_size(self):
        return int(self._L.sb2_parameter_size(self._h))

    @property
    def state_size(self):
        return int(self._L.sb2_state_size(self._h))

    # -- parameters ----------------------------------------------------------------------------------------------------
    def set_region_parameter(self, p):
        p = f64(p)
        self._ck(self._L.sb2_set_region_parameter(self._h, dptr(p), C.c_int(p.size)))

    def get_region_parameter(self):
        p = np.zeros(self.parameter_size)
        self._ck(self._L.sb2_get_region_parameter(self._h, dptr(p), C.c_int(p.size)))
        return p

    def set_catchment_parameter(self, cid, p):
        p = f64(p)
        self._ck(self._L.sb2_set_catchment_parameter(self._h, C.c_int64(cid), dptr(p), C.c_int(p.size)))

    def get_catchment_parameter(self, cid):
        p = np.zeros(self.parameter_size)
        self._ck(self._L.sb2_get_catchment_parameter(self._h, C.c_int64(cid), dptr(p), C.c_int(p.size)))
        return p

    def remove_catchment_parameter(self, cid):
        self._ck(self._L.sb2_remove_catchment_parameter(self._h, C.c_int64(cid)))

    def has_catchment_parameter(self, cid):
        return bool(self._L.sb2_has_catchment_parameter(self._h, C.c_int64(cid)))

    def set_catchment_calculation_filter(self, cids):
        a = np.ascontiguousarray(cids, dtype=np.int64)
        self._ck(self._L.sb2_set_catchment_calculation_filter(self._h, a.ctypes.data_as(capi.c_i64p), C.c_int(a.size)))

    # -- state ---------------------------------------------------------------------------------------------------------
    def set_states(self, states):
        s = f64(states)
        if s.ndim != 2:
            raise RuntimeError("states must be [cell][state_size]")
        if s.shape[0] != self.size():
            raise RuntimeError("Length of the state vector must equal number of cells")   # core/region_model.h:803-804
        if s.shape[1] != self.state_size:
            raise RuntimeError("state rows must have state_size values")
        self._ck(self._L.sb2_set_states(self._h, dptr(s), C.c_int64(s.shape[0])))

    def distribute_snow(self, states):
        """hbv_snow::state::distribute(parameter, force=False) for a flat state array: rows whose ten snow bins are all zero (the
        flat spelling of HbvSnowState(swe, sca)) get sp / sw from swe and sca, as pt_hs_k::run / run_hbv_stack do first thing
        (core/pt_hs_k.h:230, core/hbv_stack.h:312, core/hbv_snow_common.h:44-67).  -> a new [cell][state_size] array for set_states."""
        s = f64(states).copy()
        if s.shape != (self.size(), self.state_size):
            raise RuntimeError("states must be [cell][state_size]")
        self._ck(self._L.sb2_hbv_distribute_snow(self._h, dptr(s), C.c_int64(s.shape[0])))
        return s

    def get_states(self, out=None):
        """-> [cell][state_size]; `out` = a caller-owned C-contiguous float64 array of that shape to fill instead (e.g. pinned host memory)"""
        s = np.zeros((self.size(), self.state_size)) if out is None else self._checked_out(out, (self.size(), self.state_size))
        self._ck(self._L.sb2_get_states(self._h, dptr(s), C.c_int64(s.shape[0])))
        return s

    @staticmethod
    def _checked_out(out, shape):
        if not (isinstance(out, np.ndarray) and out.dtype == np.float64 and out.flags.c_contiguous and out.shape == tuple(shape)):
            raise RuntimeError(f"out must be a C-contiguous float64 array of shape {tuple(shape)}")
        return out

    current_state = property(lambda self: self.get_states())

    @property
    def initial_state(self):
        s = np.zeros((self.size(), self.state_size))
        self._ck(self._L.sb2_get_initial_state(self._h, dptr(s), C.c_int64(s.shape[0])))
        return s

    @initial_state.setter
    def initial_state(self, states):
        s = f64(states)
        if s.shape != (self.size(), self.state_size):
            raise RuntimeError("initial_state must be [cell][state_size]")
        self._ck(self._L.sb2_set_initial_state(self._h, dptr(s), C.c_int64(s.shape[0])))

    def revert_to_initial_state(self):
        self._ck(self._L.sb2_revert_to_initial_state(self._h))

    def adjust_q(self, q_scale, cids=()):
        a = np.ascontiguousarray(cids, dtype=np.int64)
        self._ck(self._L.sb2_adjust_q(self._h, C.c_double(q_scale), a.ctypes.data_as(capi.c_i64p), C.c_int(a.size)))

    def adjust_state_to_target_flow(self, wanted_flow_m3s, cids=(), start_step=0, scale_range=3.0, scale_eps=1.0e-3, max_iter=300, n_steps=1):
        """region_model::adjust_state_to_target_flow (core/region_model.h:626-637; api/boostpython/expose.h:380): -> q_adjust_result
        with .q_0, .q_r, .diagnostics; the current state is left adjusted, initial state and calculation filter are kept."""
        a = np.ascontiguousarray(cids, dtype=np.int64)
        r = capi.QAdjustResult()
        self._ck(self._L.sb2_adjust_state_to_target_flow(self._h, C.c_double(wanted_flow_m3s), a.ctypes.data_as(capi.c_i64p), C.c_int(a.size),
                                                         C.c_int64(start_step), C.c_double(scale_range), C.c_double(scale_eps), C.c_int64(max_iter),
                                                         C.c_int64(n_steps), C.byref(r)))
        return r

    def set_state_collection(self, catchment_id, on_or_off):
        # the device collects a series for all cells or for none; per-catchment switching (:844-849) selects all
        self._state_collection = bool(on_or_off)
        self._apply_collect()

    def set_snow_sca_swe_collection(self, catchment_id, on_or_off):
        self._snow_collection = bool(on_or_off)
        self._apply_collect()

    # -- environment ---------------------------------------------------------------------------------------------------
    def initialize_cell_environment(self, time_axis):
        self._ck(self._L.sb2_initialize_cell_environment(self._h, C.c_int64(time_axis.start * USEC), C.c_int64(time_axis.delta_t * USEC),
                                                         C.c_int64(time_axis.n)))
        self.time_axis = time_axis

    def set_cell_forcing(self, name, values, layout=capi.TIME_MAJOR):
        v = f64(values)
        if v.shape != ((self.time_axis.n, self.size()) if layout == capi.TIME_MAJOR else (self.size(), self.time_axis.n)):
            raise RuntimeError(f"{name}: cell forcing must be [n_steps][cell] (TIME_MAJOR) or [cell][n_steps] (CELL_MAJOR)")
        self._ck(self._L.sb2_set_cell_forcing(self._h, C.c_int(FORCING_NAMES.index(name)), dptr(v), C.c_int(layout)))

    def cell_forcing(self, name, start_step=0, n_steps=None, layout=capi.TIME_MAJOR):
        n_steps = self.time_axis.n - start_step if n_steps is None else n_steps
        out = np.zeros((n_steps, self.size()) if layout == capi.TIME_MAJOR else (self.size(), n_steps))
        self._ck(self._L.sb2_get_cell_forcing(self._h, C.c_int(FORCING_NAMES.index(name)), C.c_int64(start_step), C.c_int64(n_steps), dptr(out),
                                              C.c_int(layout)))
        return out

    def _set_sources(self, env):
        for vi, name in enumerate(FORCING_NAMES):
            src = getattr(env, name)
            if src is None:
                self._ck(self._L.sb2_set_sources(self._h, C.c_int(vi), C.c_int64(0), None, None))
                continue
            if isinstance(src, GeoPointSources):
                if src.values.shape != (src.times_us.size, src.xyz.shape[0]):
                    raise RuntimeError(f"{name}: source values must be [n_points][n_sources]")
                self._ck(self._L.sb2_set_sources_on_axis(self._h, C.c_int(vi), C.c_int64(src.xyz.shape[0]), dptr(src.xyz), C.c_int64(src.times_us.size),
                                                         src.times_us.ctypes.data_as(capi.c_i64p), C.c_int64(src.t_end_us), dptr(src.values),
                                                         C.c_int(1 if src.point_fx == "instant" else 0)))
                continue
            if isinstance(src, GeoPointSourceVector):
                self._ck(self._L.sb2_set_sources_on_axes(self._h, C.c_int(vi), C.c_int64(src.xyz.shape[0]), dptr(src.xyz),
                                                         src.n_points.ctypes.data_as(capi.c_i64p), src.times_us.ctypes.data_as(capi.c_i64p),
                                                         src.t_end_us.ctypes.data_as(capi.c_i64p), dptr(src.values),
                                                         src.point_fx.ctypes.data_as(C.POINTER(C.c_int32))))
                continue
            xyz, values = f64(src[0]), f64(src[1])
            if xyz.ndim != 2 or xyz.shape[1] != 3:
                raise RuntimeError(f"{name}: source positions must be [n_sources][3]")
            if values.shape != (self.time_axis.n, xyz.shape[0]):
                raise RuntimeError(f"{name}: source values must be [n_steps][n_sources]")
            self._ck(self._L.sb2_set_sources(self._h, C.c_int(vi), C.c_int64(xyz.shape[0]), dptr(xyz), dptr(values)))
        self.region_env = env

    def sources_on_model_axis(self, name):
        """the sources of a variable as projected onto the model axis: [n_steps][n_sources]"""
        vi = FORCING_NAMES.index(name)
        src = getattr(self.region_env, name)
        n_src = (src.xyz if isinstance(src, (GeoPointSources, GeoPointSourceVector)) else f64(src[0])).shape[0]
        out = np.zeros((self.time_axis.n, n_src))
        self._ck(self._L.sb2_get_sources_on_model_axis(self._h, C.c_int(vi), dptr(out)))
        return out

    def interpolate(self, ip_parameter, env, best_effort=True):
        self._set_sources(env)
        ok = C.c_int(0)
        self._ck(self._L.sb2_interpolate(self._h, C.byref(ip_parameter), C.c_int(1 if best_effort else 0), C.byref(ok)))
        self.ip_parameter = ip_parameter
        return bool(ok.value)

    def run_interpolation(self, ip_parameter, time_axis, env, best_effort=True):
        self.initialize_cell_environment(time_axis)
        return self.interpolate(ip_parameter, env, best_effort)

    def is_cell_env_ts_ok(self):
        ok = C.c_int(0)
        self._ck(self._L.sb2_is_cell_env_ts_ok(self._h, C.byref(ok)))
        return bool(ok.value)

    # -- the hot path ----------------------------------------------------------------------------------------------------
    def run_cells(self, use_ncore=0, start_step=0, n_steps=0):
        self._ck(self._L.sb2_run_cells(self._h, C.c_int(start_step), C.c_int(n_steps)))

    def run_windowed(self, ip_parameter, time_axis=None, env=None, start_step=0, n_steps=0, window_steps=512):
        """run_interpolation + run_cells window by window (axes whose [t][cell] forcing does not fit in HBM)."""
        if time_axis is not None:
            self.initialize_cell_environment(time_axis)
        if env is not None:
            self._set_sources(env)
        self._ck(self._L.sb2_run_windowed(self._h, C.byref(ip_parameter), C.c_int(start_step), C.c_int(n_steps), C.c_int(window_steps)))
        self.ip_parameter = ip_parameter

    def run_ensemble(self, ip_parameter, members, start_step=0, n_steps=0, window_steps=4096):
        """Interpolate and step every member of a forcing ensemble (a list of RegionEnvironment) in one device pass, from the current
        state -> (discharge, charge), each [member][n_steps][n_catchment] (n_steps == 0: the whole axis).

        Member e equals, bit for bit, setting member e's sources, interpolate(ip_parameter, env, best_effort=False), run_cells(0,
        start_step, n_steps) from the same state and reading catchment_discharges / catchment_charges of those rows.  Per variable,
        every member gives a (xyz, values [T][S]) tuple with the same xyz, or a GeoPointSources with the same xyz, times, t_end and
        point_fx; or every member leaves it None, and the model's own sources serve all members.  The model is left as it was."""
        members = list(members)
        if not members:
            raise RuntimeError("run_ensemble: no members")
        if self.time_axis is None:
            raise RuntimeError("initialize_cell_environment has not been called")
        E, T = len(members), self.time_axis.n
        for vi in range(len(FORCING_NAMES)):   # every variable's earlier ensemble sources go first: the member counts must agree
            self._ck(self._L.sb2_set_ensemble_sources(self._h, C.c_int(vi), C.c_int64(0), C.c_int64(0), None, None))
        for vi, name in enumerate(FORCING_NAMES):
            srcs = [getattr(env, name) for env in members]
            if all(s is None for s in srcs):
                continue
            if all(isinstance(s, GeoPointSources) for s in srcs):
                s0 = srcs[0]
                if not all(np.array_equal(s.xyz, s0.xyz) and np.array_equal(s.times_us, s0.times_us) and s.t_end_us == s0.t_end_us
                           and s.point_fx == s0.point_fx and s.values.shape == (s0.times_us.size, s0.xyz.shape[0]) for s in srcs):
                    raise RuntimeError(f"{name}: every member needs the same stations, times, t_end and point_fx, values [n_points][n_sources]")
                values = np.ascontiguousarray(np.stack([s.values for s in srcs]))
                self._ck(self._L.sb2_set_ensemble_sources_on_axis(self._h, C.c_int(vi), C.c_int64(E), C.c_int64(s0.xyz.shape[0]), dptr(s0.xyz),
                                                                  C.c_int64(s0.times_us.size), s0.times_us.ctypes.data_as(capi.c_i64p),
                                                                  C.c_int64(s0.t_end_us), dptr(values), C.c_int(1 if s0.point_fx == "instant" else 0)))
            elif all(isinstance(s, tuple) and len(s) == 2 for s in srcs):
                xyz = f64(srcs[0][0])
                if xyz.ndim != 2 or xyz.shape[1] != 3 or not all(np.array_equal(f64(s[0]), xyz) for s in srcs):
                    raise RuntimeError(f"{name}: every member needs the same source positions [n_sources][3]")
                if not all(np.shape(s[1]) == (T, xyz.shape[0]) for s in srcs):
                    raise RuntimeError(f"{name}: source values must be [n_steps][n_sources] in every member")
                values = np.ascontiguousarray(np.stack([f64(s[1]) for s in srcs]))
                self._ck(self._L.sb2_set_ensemble_sources(self._h, C.c_int(vi), C.c_int64(E), C.c_int64(xyz.shape[0]), dptr(xyz), dptr(values)))
            else:
                raise RuntimeError(f"{name}: the members must all give (xyz, values) tuples, all GeoPointSources, or all None")
        count = max(0, n_steps if n_steps > 0 else T)
        q = np.zeros((E, count, self.number_of_catchments()))
        c = np.zeros_like(q)
        self._ck(self._L.sb2_run_ensemble(self._h, C.byref(ip_parameter), C.c_int(start_step), C.c_int(n_steps), C.c_int(window_steps), dptr(q),
                                          dptr(c)))
        self.ip_parameter = ip_parameter
        return q, c

    # -- results -----------------------------------------------------------------------------------------------------------
    def response(self, name, start_step=0, n_steps=None, layout=capi.TIME_MAJOR):
        """cell.rc.<name> for all cells: [n_steps][cell] (or [cell][n_steps])."""
        n_steps = self.time_axis.n - start_step if n_steps is None else n_steps
        out = np.zeros((n_steps, self.size()) if layout == capi.TIME_MAJOR else (self.size(), n_steps))
        self._ck(self._L.sb2_get_response(self._h, C.c_int(RESPONSE_NAMES.index(name)), C.c_int64(start_step), C.c_int64(n_steps), dptr(out),
                                          C.c_int(layout)))
        return out

    def state_series(self, name, start_step=0, n_points=None, layout=capi.TIME_MAJOR):
        """cell.sc.<name> for all cells, T+1 instant points."""
        n_points = self.time_axis.n + 1 - start_step if n_points is None else n_points
        out = np.zeros((n_points, self.size()) if layout == capi.TIME_MAJOR else (self.size(), n_points))
        self._ck(self._L.sb2_get_state_series(self._h, C.c_int(STATE_SERIES_NAMES[self.stack].index(name)), C.c_int64(start_step),
                                              C.c_int64(n_points), dptr(out), C.c_int(layout)))
        return out

    def catchment_discharges(self, start_step=0, n_steps=None, out=None):
        n_steps = self.time_axis.n - start_step if n_steps is None else n_steps
        shape = (n_steps, self.number_of_catchments())
        out = np.zeros(shape) if out is None else self._checked_out(out, shape)
        self._ck(self._L.sb2_catchment_discharges(self._h, C.c_int64(start_step), C.c_int64(n_steps), dptr(out)))
        return out

    def catchment_charges(self, start_step=0, n_steps=None):
        n_steps = self.time_axis.n - start_step if n_steps is None else n_steps
        out = np.zeros((n_steps, self.number_of_catchments()))
        self._ck(self._L.sb2_catchment_charges(self._h, C.c_int64(start_step), C.c_int64(n_steps), dptr(out)))
        return out

    # -- routing -------------------------------------------------------------------------------------------------------------
    def set_river_network(self, rivers):
        """rivers [n][6] = id, downstream id, downstream distance, uhg velocity, alpha, beta (routing.h:98-123)."""
        r = f64(rivers).reshape(-1, 6)
        self._ck(self._L.sb2_set_river_network(self._h, C.c_int64(r.shape[0]), dptr(r)))

    def _river(self, rid, which):
        n = self.time_axis.n
        out = [np.zeros(n) if which == k else None for k in range(3)]
        self._ck(self._L.sb2_river_flows(self._h, C.c_int64(rid), C.c_int64(0), C.c_int64(n), dptr(out[0]), dptr(out[1]), dptr(out[2])))
        return out[which]

    def river_local_inflow_m3s(self, rid):
        return self._river(rid, 0)

    def river_upstream_inflow_m3s(self, rid):
        return self._river(rid, 1)

    def river_output_flow_m3s(self, rid):
        return self._river(rid, 2)

    # -- device-side hooks -------------------------------------------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self._L.sb2_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def set_idw_dense(self, on):
        """IDW as a dense tensor-core contraction when all station values are finite (default on); off = per-neighbour kernel."""
        self._ck(self._L.sb2_set_idw_dense(self._h, C.c_int(1 if on else 0)))

    def kernel_launches(self):
        return int(self._L.sb2_kernel_launches(self._h))

    def step_chunk_steps(self):
        """steps one launch of the step kernels covers (a forcing window is stepped in chunks of this many steps)"""
        return int(self._L.sb2_step_chunk_steps(self._h))

    def last_run_kernel_ms(self):
        a, b = C.c_float(0), C.c_float(0)
        self._ck(self._L.sb2_last_run_kernel_ms(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def device_catchment_discharges(self):
        p, t, k = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        self._ck(self._L.sb2_device_catchment_discharges(self._h, C.byref(p), C.byref(t), C.byref(k)))
        return p.value, t.value, k.value

    def device_catchment_charges(self):
        p, t, k = C.c_void_p(), C.c_int64(0), C.c_int64(0)
        self._ck(self._L.sb2_device_catchment_charges(self._h, C.byref(p), C.byref(t), C.byref(k)))
        return p.value, t.value, k.value


class PTGSKModel(RegionModel):
    """PTGSKModel with the statistics properties of shyft/api/pt_gs_k/__init__.py:14-20"""
    stack = PT_GS_K
    gamma_snow_state = property(lambda self: _stats().GammaSnowStateStatistics(self))
    gamma_snow_response = property(lambda self: _stats().GammaSnowResponseStatistics(self))
    priestley_taylor_response = property(lambda self: _stats().PriestleyTaylorResponseStatistics(self))
    actual_evaptranspiration_response = property(lambda self: _stats().ActualEvapotranspirationResponseStatistics(self))
    kirchner_state = property(lambda self: _stats().KirchnerStateStatistics(self))


class PTGSKOptModel(RegionModel):  # cell_discharge_response_t: discharge_collector + null state collector
    stack = PT_GS_K
    default_collect = COLLECT_DISCHARGE


class PTHSKModel(RegionModel):
    """PTHSKModel with the statistics properties of shyft/api/pt_hs_k/__init__.py:13-19"""
    stack = PT_HS_K
    hbv_snow_state = property(lambda self: _stats().HbvSnowStateStatistics(self))
    hbv_snow_response = property(lambda self: _stats().HbvSnowResponseStatistics(self))
    priestley_taylor_response = property(lambda self: _stats().PriestleyTaylorResponseStatistics(self))
    actual_evaptranspiration_response = property(lambda self: _stats().ActualEvapotranspirationResponseStatistics(self))
    kirchner_state = property(lambda self: _stats().KirchnerStateStatistics(self))


class PTHSKOptModel(RegionModel):
    stack = PT_HS_K
    default_collect = COLLECT_DISCHARGE


class PTSSKModel(RegionModel):
    """PTSSKModel (shyft/api/pt_ss_k/__init__.py): Priestley-Taylor, Skaugen snow, actual evapotranspiration, Kirchner"""
    stack = PT_SS_K
    priestley_taylor_response = property(lambda self: _stats().PriestleyTaylorResponseStatistics(self))
    actual_evaptranspiration_response = property(lambda self: _stats().ActualEvapotranspirationResponseStatistics(self))
    kirchner_state = property(lambda self: _stats().KirchnerStateStatistics(self))


class PTSSKOptModel(RegionModel):
    stack = PT_SS_K
    default_collect = COLLECT_DISCHARGE


class PTHPSKModel(RegionModel):
    """PTHPSKModel (shyft/api/pt_hps_k/__init__.py): Priestley-Taylor, hbv_physical_snow, actual evapotranspiration, Kirchner"""
    stack = PT_HPS_K
    priestley_taylor_response = property(lambda self: _stats().PriestleyTaylorResponseStatistics(self))
    actual_evaptranspiration_response = property(lambda self: _stats().ActualEvapotranspirationResponseStatistics(self))
    kirchner_state = property(lambda self: _stats().KirchnerStateStatistics(self))


class PTHPSKOptModel(RegionModel):
    stack = PT_HPS_K
    default_collect = COLLECT_DISCHARGE


class HbvStackModel(RegionModel):
    """HbvModel with the statistics properties of shyft/api/hbv_stack/__init__.py:13-19"""
    stack = HBV_STACK
    hbv_snow_state = property(lambda self: _stats().HbvSnowStateStatistics(self))
    hbv_snow_response = property(lambda self: _stats().HbvSnowResponseStatistics(self))
    priestley_taylor_response = property(lambda self: _stats().PriestleyTaylorResponseStatistics(self))
    hbv_actual_evaptranspiration_response = property(lambda self: _stats().HbvActualEvapotranspirationResponseStatistics(self))
    soil_state = property(lambda self: _stats().HbvSoilStateStatistics(self))
    soil_response = property(lambda self: _stats().HbvSoilResponseStatistics(self))
    tank_state = property(lambda self: _stats().HbvTankStateStatistics(self))


HbvModel, HbvOptModel = HbvStackModel, None  # the reference's Python names (shyft/api/hbv_stack/__init__.py); HbvOptModel bound below


class HbvStackOptModel(RegionModel):
    stack = HBV_STACK
    default_collect = COLLECT_DISCHARGE


HbvOptModel = HbvStackOptModel
