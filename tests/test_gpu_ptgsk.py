"""GPU parity of the pt_gs_k hot path: every call goes through the C ABI (shyft_b200/libshyft_b200.so); the oracle is the checker.

Tolerance (north_star): state and discharge within 1e-9 relative per time step; catchment / cell indexing bit-exact.
"""
import json
import os

import numpy as np
import pytest

from fixtures import FORCING, PTGSK_DEFAULT, geo_matrix, oracle_interpolate_py_fixture, py_region_fixture
from parity import assert_parity

pytestmark = pytest.mark.gpu
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_known_answers.json")))["region_pt_gs_k_20x240"]


def _model_from_py_fixture(sb, fx, cls=None):
    cls = cls or sb.PTGSKModel
    g = fx["geo"]
    geo = sb.geo_cell_data_vector(g[:, 0], g[:, 1], g[:, 2], g[:, 3], g[:, 4].astype(np.int64), g[:, 5], g[:, 6], g[:, 7], g[:, 8], g[:, 9])
    m = cls(geo, fx["par"])
    ta = sb.TimeAxis(fx["t0"], fx["dt"], fx["T"])
    xyz = fx["station"][None, :]
    env = sb.RegionEnvironment(**{k: (xyz, np.full((fx["T"], 1), v)) for k, v in fx["consts"].items()})
    return m, ta, env


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def test_reference_region_fixture_literals_and_oracle(sb, oracle):
    """The reference's own 20 cells x 240 h region (test_region_model_stacks.py:145-304) through the C ABI."""
    fx = py_region_fixture()
    m, ta, env = _model_from_py_fixture(sb, fx)
    ip = sb.InterpolationParameter()
    ip.use_idw_for_temperature = 1
    ip.temperature_idw.default_temp_gradient = -0.005
    ip.temperature_idw.gradient_by_equation = 1
    ip.temperature_idw.max_members = 6
    ip.temperature_idw.max_distance = 20000
    ip.temperature_idw.zscale = 0.5
    ip.temperature_idw.distance_measure_factor = 1.0
    m.initialize_cell_environment(ta)
    assert m.interpolate(ip, env)
    assert m.is_cell_env_ts_ok()
    f_oracle = oracle_interpolate_py_fixture(oracle, fx)
    for name in FORCING:
        assert_parity(m.cell_forcing(name), f_oracle[name], "env_ts." + name, rtol=1e-14)
    m.set_states(fx["state"])
    m.set_state_collection(-1, True)
    m.run_cells()
    want = oracle.ptgsk_run_cells(fx["geo"], fx["par"], f_oracle, fx["state"], fx["t0"] * 10**6, fx["dt"] * 10**6, collect_response=True,
                                  collect_state=True)
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert_parity(m.response(name), want[name], name)
    for name in sb.capi.STATE_SERIES_NAMES[sb.PT_GS_K]:
        assert_parity(m.state_series(name), want[name], name)
    assert_parity(m.get_states(), want["state"], "end state")
    # the reference's literals, straight from the GPU results
    ch = m.response("charge_m3s")
    assert ch[0].sum() == pytest.approx(GOLD["charge_sum_step0"]["value"], abs=1e-4)
    assert ch[0, [0, 1, 3]].sum() == pytest.approx(GOLD["charge_cells_0_1_3_step0"]["value"], abs=1e-4)
    assert ch[:, [1, 2, 6]].sum() == pytest.approx(GOLD["charge_sum_cells_1_2_6_all_steps"]["value"], abs=2e-4)
    assert m.response("ae_output").mean(axis=1).max() == pytest.approx(GOLD["ae_output_max"]["value"], abs=1e-12)
    q_mmh = m.state_series("kirchner_discharge") / (fx["geo"][:, 3] / 3.6e6)
    assert (1.0 - np.exp(-q_mmh * 3.0 / fx["par"][3])).mean(axis=1).min() == pytest.approx(GOLD["ae_pot_ratio_min"]["value"], abs=1e-12)
    cd = m.catchment_discharges()
    assert cd.shape == (240, 1) and cd[0, 0] >= GOLD["discharge_step0_min"]
    assert_parity(cd[:, 0], want["avg_discharge"].sum(axis=1), "catchment discharge", rtol=1e-12)
    # routing: river 1, 3000 m at 1/3.6 m/s -> 3-step gamma unit hydrograph
    g = m.geo.copy()
    g["routing_id"] = 1
    m2 = sb.PTGSKModel(g, fx["par"])
    m2.initialize_cell_environment(ta)
    m2.interpolate(ip, env)
    m2.set_states(fx["state"])
    m2.run_cells()
    m2.set_river_network([[1, 0, 3000.0, 1 / 3.60, 7.0, 0.0]])
    out = m2.river_output_flow_m3s(1)
    assert out[8] == pytest.approx(GOLD["river_out_value_8"]["value"], abs=1e-10)
    assert np.all(m2.river_upstream_inflow_m3s(1) == 0.0)
    assert_parity(m2.river_local_inflow_m3s(1), want["avg_discharge"].sum(axis=1), "river local inflow", rtol=1e-12)


def test_chunked_run_is_bit_identical_to_one_shot(sb):
    fx = py_region_fixture()
    m, ta, env = _model_from_py_fixture(sb, fx)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    m.run_interpolation(ip, ta, env)
    m.set_states(fx["state"])
    m.run_cells()
    q1, s1 = m.response("avg_discharge"), m.get_states()
    m.revert_to_initial_state()
    m.run_interpolation(ip, ta, env)  # fresh axis -> fresh, NaN-filled series (cell_model.h:163-170)
    for k in range(10):
        m.run_cells(0, 24 * k, 24)
        if k < 9:
            assert np.all(np.isnan(m.response("avg_discharge", 24 * (k + 1), 24)))
    assert np.array_equal(m.response("avg_discharge"), q1)
    assert np.array_equal(m.get_states(), s1)


def _synthetic(sb, n_cells, n_steps, n_stations, **kw):
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n_cells, n_steps, n_stations, **kw)
    return geo, ta, env, synthetic.default_state(0, n_cells)


def _oracle_forcing(oracle, geo, ta, env, ip_idw=True):
    gm = geo_matrix(geo)
    dst = gm[:, :3]
    f = {}
    for name in FORCING:
        xyz, vals = getattr(env, name)
        vals = oracle.average_accessor_same_axis(vals, ta.delta_t * 10**6)
        if name == "temperature" and not ip_idw:
            f[name] = oracle.btk_run(xyz, vals, dst, ta.start * 10**6, ta.delta_t * 10**6)
        else:
            mm = 20 if name in ("temperature", "precipitation") else 10
            f[name] = oracle.idw_run(name, xyz, vals, dst, oracle.idw_par(max_members=mm), dst_slope=gm[:, 5], ncore=8)
    return gm, f


@pytest.mark.parametrize("collect,n", [("all+state", 256), ("discharge", 1000)])
def test_config1_slice_parity_through_a_winter(sb, oracle, collect, n):
    """BASELINE configs[0] (1 000 synthetic cells x 1 year hourly, IDW interpolation, discharge collector) in full, and 256 cells of it
    with every response and state series collected: each series and the end state against the oracle, step by step."""
    T, S = 8760, 16
    geo, ta, env, st0 = _synthetic(sb, n, T, S, config_index=0, cells_per_catchment=100)
    m = (sb.PTGSKModel if collect == "all+state" else sb.PTGSKOptModel)(geo, PTGSK_DEFAULT)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    assert m.run_interpolation(ip, ta, env)
    gm, f = _oracle_forcing(oracle, geo, ta, env, ip_idw=True)
    for name in FORCING:
        assert_parity(m.cell_forcing(name), f[name], "env_ts." + name, rtol=1e-12)
    # run both from the SAME forcing bits so that the cell-stack comparison is not blurred by interpolation round-off
    for name in FORCING:
        m.set_cell_forcing(name, f[name])
    m.set_states(st0)
    if collect == "all+state":
        m.set_state_collection(-1, True)
    m.run_cells()
    want = oracle.ptgsk_run_cells(gm, PTGSK_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, collect_response=True, collect_state=True,
                                  ncore=8)
    assert np.nanmax(want["snow_swe"]) > 10.0, "the fixture must build a snow pack"
    names = ("avg_discharge", "charge_m3s") if collect == "discharge" else \
        ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output")
    for name in names:
        assert_parity(m.response(name), want[name], name)
    if collect == "all+state":
        for name in sb.capi.STATE_SERIES_NAMES[sb.PT_GS_K]:
            assert_parity(m.state_series(name), want[name], name)
    assert_parity(m.get_states(), want["state"], "end state")
    # one operation sequence on both machines (DESIGN.md "Deterministic math"): the per-cell results are in fact bit-identical
    for name in names:
        assert np.array_equal(m.response(name), want[name], equal_nan=True), name + " is within 1e-9 but not bit-identical"
    assert np.array_equal(m.get_states(), want["state"])
    cix = m.cell_catchment_ix()
    cq = m.catchment_discharges()
    for k in range(m.number_of_catchments()):
        assert_parity(cq[:, k], want["avg_discharge"][:, cix == k].sum(axis=1), f"catchment {k} discharge", rtol=1e-12)
    cc = m.catchment_charges()
    for k in range(m.number_of_catchments()):
        assert_parity(cc[:, k], want["charge_m3s"][:, cix == k].sum(axis=1), f"catchment {k} charge", rtol=1e-9, atol_frac=1e-12)


@pytest.mark.parametrize("n,T", [(1, 1), (1, 130), (31, 63), (31, 127), (33, 65), (33, 128), (100, 129), (257, 1)])
def test_ragged_sizes_are_bit_identical(sb, oracle, n, T):
    """One cell, one step, cell counts around a warp and step counts around the 128-step slice of the time split: every series and
    the end state equal the oracle's bit for bit (out-of-range lanes of the last warp shadow a cell and store nothing)."""
    geo, ta, env, st0 = _synthetic(sb, n, T, 4, config_index=30 + n % 7, cells_per_catchment=max(1, n // 3), start=1424476800)  # 2015-02-21
    st0[:, 5] = -1.0                      # acc_melt < 0: accumulation branch
    st0[:, 4] = np.linspace(5.0, 80.0, n)  # sdc_melt_mean: a snow pack from the first step on
    st0[:, 1] = 2.0                       # some liquid water: wet-snow paths, Brent on snowfall
    m = sb.PTGSKModel(geo, PTGSK_DEFAULT)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    assert m.run_interpolation(ip, ta, env)
    gm, f = _oracle_forcing(oracle, geo, ta, env, ip_idw=True)
    for name in FORCING:
        m.set_cell_forcing(name, f[name])
    m.set_states(st0)
    m.set_state_collection(-1, True)
    m.run_cells()
    want = oracle.ptgsk_run_cells(gm, PTGSK_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, collect_response=True, collect_state=True, ncore=2)
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert np.array_equal(m.response(name), want[name], equal_nan=True), name
    for name in sb.capi.STATE_SERIES_NAMES[sb.PT_GS_K]:
        assert np.array_equal(m.state_series(name), want[name], equal_nan=True), name
    assert np.array_equal(m.get_states(), want["state"])
    assert m.catchment_discharges().shape == (T, m.number_of_catchments())
    assert np.allclose(m.catchment_discharges().sum(axis=1), want["avg_discharge"].sum(axis=1), rtol=1e-12)


def test_catchment_indexing_is_bit_exact(sb, oracle):
    rng = np.random.default_rng(5)
    cids = rng.integers(1, 40, 777) * 13
    geo = sb.geo_cell_data_vector(np.arange(777.0), np.zeros(777), np.zeros(777), catchment_id=cids)
    m = sb.PTGSKOptModel(geo)
    cix, ids = oracle.catchment_index(cids)
    assert np.array_equal(m.cell_catchment_ix(), cix)
    assert np.array_equal(m.catchment_ids, ids)


def test_windowed_run_equals_resident_run(sb):
    n, T, S = 300, 1200, 9
    geo, ta, env, st0 = _synthetic(sb, n, T, S, config_index=7, cells_per_catchment=64, start=1417392000)  # 2014-12-01
    ip = sb.InterpolationParameter()  # BTK temperature + IDW
    a = sb.PTGSKOptModel(geo, PTGSK_DEFAULT)
    a.run_interpolation(ip, ta, env)
    a.set_states(st0)
    a.run_cells()
    b = sb.PTGSKOptModel(geo, PTGSK_DEFAULT)
    b.initialize_cell_environment(ta)
    b.set_states(st0)
    b.run_windowed(ip, env=env, window_steps=250)
    assert np.array_equal(a.catchment_discharges(), b.catchment_discharges())
    assert np.array_equal(a.get_states(), b.get_states())
    assert np.array_equal(a.response("avg_discharge", 1000, 200), b.response("avg_discharge", 1000, 200))  # the last window is resident


def test_catchment_parameters_filter_and_errors(sb, oracle):
    n, T, S = 96, 240, 4
    geo, ta, env, st0 = _synthetic(sb, n, T, S, config_index=3, cells_per_catchment=32, start=1422748800)  # 2015-02-01
    m = sb.PTGSKModel(geo, PTGSK_DEFAULT)
    with pytest.raises(RuntimeError, match="region_model::run with invalid time_axis invoked"):
        m.run_cells()
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    m.run_interpolation(ip, ta, env)
    with pytest.raises(RuntimeError, match=r"start_step must in range"):
        m.run_cells(0, T, 1)
    with pytest.raises(RuntimeError, match="n_steps must be range"):
        m.run_cells(0, 0, -1)
    with pytest.raises(RuntimeError, match=r"start_step\+n_steps must be within time-axis range"):
        m.run_cells(0, 10, T)
    with pytest.raises(RuntimeError, match="Length of the state vector must equal number of cells"):
        m.set_states(st0[:-1])
    with pytest.raises(RuntimeError, match="no cells have supplied cid"):
        m.set_catchment_calculation_filter([99])
    with pytest.raises(RuntimeError, match="Initial state not yet established or set"):
        m.revert_to_initial_state()
    # catchment 2 gets its own parameter set (region_model.h:668-678)
    p2 = PTGSK_DEFAULT.copy()
    p2[0], p2[4], p2[16] = -2.9, 0.5, 1.2
    m.set_catchment_parameter(2, p2)
    assert m.has_catchment_parameter(2) and not m.has_catchment_parameter(1)
    assert np.array_equal(m.get_catchment_parameter(2), p2) and np.array_equal(m.get_catchment_parameter(1), PTGSK_DEFAULT)
    m.set_states(st0)
    m.run_cells()
    gm = geo_matrix(geo)
    f = {k: m.cell_forcing(k) for k in FORCING}
    pset = (gm[:, 4] == 2).astype(np.int32)
    want = oracle.ptgsk_run_cells(gm, np.stack([PTGSK_DEFAULT, p2]), f, st0, ta.start * 10**6, ta.delta_t * 10**6, pset_of_cell=pset)
    assert_parity(m.response("avg_discharge"), want["avg_discharge"], "avg_discharge with catchment parameters")
    # calculation filter: only catchment 3 is stepped, the others keep state; catchment sums of the others are 0 (:873-885)
    m.revert_to_initial_state()
    m.set_catchment_calculation_filter([3])
    m.run_cells()
    s = m.get_states()
    assert np.array_equal(s[gm[:, 4] != 3], st0[gm[:, 4] != 3])
    cq = m.catchment_discharges()
    assert np.all(cq[:, [0, 1]] == 0.0) and np.all(cq[:, 2] > 0.0)
    assert_parity(m.response("avg_discharge")[:, gm[:, 4] == 3], want["avg_discharge"][:, gm[:, 4] == 3], "filtered avg_discharge")
    m.set_catchment_calculation_filter([])
    # adjust_q scales kirchner.q of the selected catchments (:831-837)
    m.revert_to_initial_state()
    m.adjust_q(2.0, [1])
    s = m.get_states()
    assert np.array_equal(s[gm[:, 4] == 1, 8], 2.0 * st0[gm[:, 4] == 1, 8]) and np.array_equal(s[gm[:, 4] != 1, 8], st0[gm[:, 4] != 1, 8])


def test_full_size_properties_config2_slice(sb):
    """Size-independent properties at a size the oracle cannot reach quickly: 20k cells x 2 years through the windowed
    path.  (i) water balance: charge integrates to the storage change implied by discharge, (ii) catchment sums equal
    the sums of the per-cell series in the resident window, (iii) rerun from the initial state is bit-identical."""
    n, T, S = 20000, 17520, 64
    geo, ta, env, st0 = _synthetic(sb, n, T, S, config_index=1)
    m = sb.PTGSKOptModel(geo, PTGSK_DEFAULT)
    m.initialize_cell_environment(ta)
    m.set_states(st0)
    ip = sb.InterpolationParameter()
    m.run_windowed(ip, env=env, window_steps=584)
    cq, cc, s1 = m.catchment_discharges(), m.catchment_charges(), m.get_states()
    assert np.all(np.isfinite(cq)) and np.all(cq >= 0.0) and np.all(np.isfinite(s1))
    last = T - 584
    cix = m.cell_catchment_ix()
    q = m.response("avg_discharge", last, 584)
    for k in range(m.number_of_catchments()):
        assert np.allclose(cq[last:, k], q[:, cix == k].sum(axis=1), rtol=1e-12, atol=0)
    # charge = precip + glacier melt - ae - discharge: summed over two years it equals the change in stored water, which is
    # bounded by the snow pack + ground water a cell can hold; it must be tiny next to the cumulated discharge
    assert abs(cc.sum()) < 0.25 * cq.sum()
    m.revert_to_initial_state()
    m.run_windowed(ip, window_steps=584)
    assert np.array_equal(m.catchment_discharges(), cq) and np.array_equal(m.get_states(), s1)


def test_time_sliced_kernels_are_deterministic_and_slicing_invariant(sb):
    """The snow / response kernels hand a window out in 128-step slices by ticket, each slice waiting for its cell group's previous
    one (sb2_ptgsk.cuh).  With several waves of blocks (60 000 cells x 5 slices) three runs must agree bit for bit, and so must a
    run cut into odd chunks (other slice boundaries, other ticket order) and a windowed run."""
    n, T = 60000, 640
    geo, ta, env, st0 = _synthetic(sb, n, T, 16, config_index=21, start=1417392000)  # 2014-12-01: snow, melt events, wet-snow snowfall
    m = sb.PTGSKOptModel(geo)
    ip = sb.InterpolationParameter()
    assert m.run_interpolation(ip, ta, env)
    m.set_states(st0)
    m.run_cells()
    q0, c0, s0 = m.catchment_discharges(), m.catchment_charges(), m.get_states()
    assert np.all(np.isfinite(q0)) and np.all(np.isfinite(s0))
    for _ in range(2):
        m.revert_to_initial_state()
        m.run_cells()
        assert np.array_equal(m.catchment_discharges(), q0) and np.array_equal(m.catchment_charges(), c0)
        assert np.array_equal(m.get_states(), s0)
    m.revert_to_initial_state()
    done = 0
    for chunk in (37, 64, 1, 200, 129, 209):
        m.run_cells(0, done, chunk)
        done += chunk
    assert done == T
    assert np.array_equal(m.catchment_discharges(), q0) and np.array_equal(m.get_states(), s0)
    m.revert_to_initial_state()
    m.run_windowed(ip, window_steps=150)
    assert np.array_equal(m.catchment_discharges(), q0) and np.array_equal(m.get_states(), s0)


def test_cpp_host_shim_selftest():
    """include/shyft_b200/region_model.hpp (the C++ mirror of region_model<cell_t>) over the C ABI, reference literals."""
    import subprocess
    from shyft_b200 import _build
    exe = _build.build_host_shim_test()
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "shim selftest ok" in r.stdout
