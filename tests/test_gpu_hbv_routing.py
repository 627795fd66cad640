"""GPU parity of the pt_hs_k and hbv_stack stacks and of river routing (BASELINE config 3 shape) through the C ABI."""
import numpy as np
import pytest

from fixtures import FORCING, HBV_DEFAULT, PTHSK_DEFAULT, geo_matrix
from parity import assert_parity

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def _setup(sb, cls, par, stack, n=320, T=6000, S=16):
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, S, config_index=2, cells_per_catchment=40, with_routing=True, start=1414800000)  # 2014-11-01
    m = cls(geo, par)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    st0 = synthetic.default_state(stack, n)
    m.set_states(st0)
    f = {k: m.cell_forcing(k) for k in FORCING}
    return m, geo, ta, st0, f


def test_pt_hs_k_parity(sb, oracle):
    m, geo, ta, st0, f = _setup(sb, sb.PTHSKModel, PTHSK_DEFAULT, 1)
    m.run_cells()
    want = oracle.pthsk_run_cells(geo_matrix(geo), PTHSK_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, ncore=8)
    assert np.nanmax(want["snow_swe"]) > 5.0
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert_parity(m.response(name), want[name], "pt_hs_k " + name)
    assert_parity(m.get_states(), want["state"], "pt_hs_k end state")
    # one operation sequence on both machines (DESIGN.md "Deterministic math"): the per-cell results are in fact bit-identical
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert np.array_equal(m.response(name), want[name], equal_nan=True), "pt_hs_k " + name + " is within 1e-9 but not bit-identical"
    assert np.array_equal(m.get_states(), want["state"])


def test_hbv_stack_parity(sb, oracle):
    m, geo, ta, st0, f = _setup(sb, sb.HbvStackModel, HBV_DEFAULT, 2)
    m.run_cells()
    want = oracle.hbv_stack_run_cells(geo_matrix(geo), HBV_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, ncore=8)
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output", "soil_outflow"):
        assert_parity(m.response(name), want[name], "hbv_stack " + name)
    assert_parity(m.get_states(), want["state"], "hbv_stack end state")
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output", "soil_outflow"):
        assert np.array_equal(m.response(name), want[name], equal_nan=True), "hbv_stack " + name + " is within 1e-9 but not bit-identical"
    assert np.array_equal(m.get_states(), want["state"])


def test_hbv_chunked_equals_one_shot_and_state_series(sb):
    m, geo, ta, st0, f = _setup(sb, sb.HbvStackModel, HBV_DEFAULT, 2, n=100, T=480)
    m.set_state_collection(-1, True)
    m.run_cells()
    q, s = m.response("avg_discharge"), m.get_states()
    sm = m.state_series("soil_moisture")
    assert np.array_equal(sm[0], st0[:, 12]) and np.array_equal(sm[-1], s[:, 12])
    m.revert_to_initial_state()
    for k in range(4):
        m.run_cells(0, 120 * k, 120)
    assert np.array_equal(m.response("avg_discharge"), q) and np.array_equal(m.get_states(), s)


def test_river_network_routing_parity(sb, oracle):
    from shyft_b200 import synthetic
    m, geo, ta, st0, f = _setup(sb, sb.PTHSKModel, PTHSK_DEFAULT, 1, n=320, T=1000)
    m.run_cells()
    rivers = synthetic.river_chain(m.number_of_catchments(), depth=4)
    m.set_river_network(rivers)
    gm = geo_matrix(geo)
    q = m.response("avg_discharge")
    uhg = np.tile(PTHSK_DEFAULT[13:16], (gm.shape[0], 1))
    for rid in (1, 4, 8):
        local, up, out = oracle.river_flows(rivers, rid, q, gm[:, 10].astype(np.int64), gm[:, 11], uhg, ta.delta_t * 10**6)
        assert_parity(m.river_local_inflow_m3s(rid), local, f"river {rid} local inflow", rtol=1e-12)
        assert_parity(m.river_upstream_inflow_m3s(rid), up, f"river {rid} upstream inflow", rtol=1e-12)
        assert_parity(m.river_output_flow_m3s(rid), out, f"river {rid} output", rtol=1e-12)
    with pytest.raises(RuntimeError, match="cycle"):
        m.set_river_network([[1, 2, 100.0, 1.0, 7.0, 0.0], [2, 1, 100.0, 1.0, 7.0, 0.0]])
    with pytest.raises(RuntimeError, match="not found"):
        m.river_output_flow_m3s(999)


@pytest.mark.parametrize("stack", ["pt_hs_k", "hbv_stack"])
def test_windowed_run_with_routing_equals_resident_run(sb, stack):
    """BASELINE config 3 shape: the axis does not fit in HBM at 400k cells, so rivers are fed window by window."""
    from shyft_b200 import synthetic
    cls, par, sid = (sb.PTHSKOptModel, PTHSK_DEFAULT, 1) if stack == "pt_hs_k" else (sb.HbvStackOptModel, HBV_DEFAULT, 2)
    n, T, S = 640, 1500, 16
    geo, ta, env = synthetic.make_region(n, T, S, config_index=2, cells_per_catchment=40, with_routing=True, start=1414800000)
    rivers = synthetic.river_chain(n // 40, depth=8)
    st0 = synthetic.default_state(sid, n)
    ip = sb.InterpolationParameter()
    a = cls(geo, par)
    a.run_interpolation(ip, ta, env)
    a.set_states(st0)
    a.set_river_network(rivers)
    a.run_cells()
    b = cls(geo, par)
    b.initialize_cell_environment(ta)
    b.set_states(st0)
    b.set_river_network(rivers)
    b.run_windowed(ip, env=env, window_steps=333)
    assert np.array_equal(a.catchment_discharges(), b.catchment_discharges())
    for rid in (1, 5, 8, 16):
        assert_parity(b.river_local_inflow_m3s(rid), a.river_local_inflow_m3s(rid), f"{stack} river {rid} local inflow (windowed)", rtol=1e-13)
        assert_parity(b.river_output_flow_m3s(rid), a.river_output_flow_m3s(rid), f"{stack} river {rid} output (windowed)", rtol=1e-13)
    assert a.river_output_flow_m3s(8).max() > a.river_local_inflow_m3s(8).max()  # the chain accumulates upstream flow


@pytest.mark.parametrize("stack", [1, 2])
def test_per_bin_snow_state_series(sb, oracle, stack):
    """state_collector of the HBV stacks (core/pt_hs_k_cell_model.h:193-205, core/hbv_stack_cell_model.h:196-212): sp[i] / sw[i] of the
    five snow bins at the beginning of every step and after the last one, against the oracle stepped one step at a time"""
    cls, par = (sb.PTHSKModel, PTHSK_DEFAULT) if stack == 1 else (sb.HbvStackModel, HBV_DEFAULT)
    m, geo, ta, st0, f = _setup(sb, cls, par, stack, n=48, T=400)
    m.set_state_collection(-1, True)
    m.run_cells()
    run = oracle.pthsk_run_cells if stack == 1 else oracle.hbv_stack_run_cells
    G = geo_matrix(geo)
    st = st0.copy()
    want = np.zeros((401, 48, 10))
    for i in range(400):
        want[i] = st[:, 2:12]
        st = run(G, par, f, st, ta.start * 10**6, ta.delta_t * 10**6, start_step=i, n_steps=1)["state"]
    want[400] = st[:, 2:12]
    assert want[:, :, :5].max() > 1.0      # there is snow in the bins
    for i in range(5):
        assert np.array_equal(m.state_series(f"snow_sp_{i}"), want[:, :, i]), i
        assert np.array_equal(m.state_series(f"snow_sw_{i}"), want[:, :, 5 + i]), i
    # the statistics readers over them (api/api.h:1086-1160): one area-weighted series / per-cell vector / value per bin
    cids, area = geo["catchment_id"], geo["area"]
    sel = [int(cids[0])]
    sp = m.hbv_snow_state.sp(sel)
    assert len(sp) == 5 and sp[0].shape == (401,)
    for i in range(5):
        assert np.allclose(sp[i], oracle.average_catchment_feature(want[:, :, i], area, cids, sel), rtol=1e-12, atol=1e-300)
        assert np.array_equal(m.hbv_snow_state.sw(sel, 200)[i], oracle.catchment_feature(want[:, :, 5 + i], cids, sel, 200))
    v = m.hbv_snow_state.sp_value(sel, 200)
    assert v == pytest.approx([oracle.average_catchment_feature_value(want[:, :, i], area, cids, sel, 200) for i in range(5)], rel=1e-12)


def test_reference_python_hbv_model_run(sb, oracle):
    """shyft/tests/api/test_region_model_stacks.py:423-480 (HbvModel): 20 cells x 240 h, one constant point source per variable given as
    a single-point series over the whole period (create_time_point_ts :31-40 -- projected on the device by average_accessor),
    IDW temperature with gradient_by_equation, default HbvState with tank.uz = tank.lz = 40; discharge_value(cids, 0) >= 32"""
    from fixtures import py_region_fixture
    fx = py_region_fixture()
    g = fx["geo"]
    geo = sb.geo_cell_data_vector(g[:, 0], g[:, 1], g[:, 2], area=g[:, 3], catchment_id=g[:, 4].astype(np.int64), radiation_slope_factor=g[:, 5],
                                  glacier=g[:, 6], lake=g[:, 7], reservoir=g[:, 8], forest=g[:, 9])
    m = sb.HbvModel(geo, HBV_DEFAULT)
    assert m.size() == 20
    ta = sb.TimeAxis(fx["t0"], 3600, 240)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    ip.temperature_idw.default_temp_gradient = -0.005
    ip.temperature_idw.gradient_by_equation = 1
    ip.temperature_idw.max_members = 6
    ip.temperature_idw.max_distance = 20000
    assert ip.temperature_idw.zscale == 1.0
    ip.temperature_idw.zscale = 0.5
    ip.temperature_idw.distance_measure_factor = 1.0
    assert ip.precipitation.scale_factor == pytest.approx(1.02)
    end = fx["t0"] + 240 * 3600
    env = sb.RegionEnvironment(**{k: sb.GeoPointSources(fx["station"][None, :], [fx["t0"]], [[v]], t_end=end, point_fx="average")
                                  for k, v in fx["consts"].items()})
    assert m.run_interpolation(ip, ta, env)
    s0 = np.zeros((20, 15))
    s0[:, 13:15] = 40.0   # HbvState(): snow 0, soil.sm 0 (hbv_soil.h:28-29), tank.uz = tank.lz = 40 as the test sets them
    m.set_states(s0)
    m.set_state_collection(-1, False)
    m.run_cells()
    q_without = m.statistics.discharge([])
    m.set_states(s0)
    m.set_state_collection(-1, True)
    m.run_cells()
    q = m.statistics.discharge([])
    assert np.array_equal(q, q_without)
    assert m.statistics.discharge_value([], 0) >= 32.0
    with pytest.raises(RuntimeError, match="does not exist"):
        m.statistics.discharge([0, 4, 5])
    # the same run on the oracle
    f = {k: m.cell_forcing(k) for k in FORCING}
    assert np.all(f["temperature"] == 10.0) and np.allclose(f["radiation"], 300.0 * 0.9)   # single-source copy / slope factor
    want = oracle.hbv_stack_run_cells(g, HBV_DEFAULT, f, s0, fx["t0"] * 10**6, 3600 * 10**6)
    assert_parity(m.response("avg_discharge"), want["avg_discharge"], "hbv python fixture discharge")
    assert want["avg_discharge"][0].sum() >= 32.0


@pytest.mark.parametrize("stack", [1, 2])
def test_snow_state_given_as_swe_and_sca_is_distributed_like_the_reference(sb, oracle, stack):
    """HbvSnowState(swe, sca) with empty bins: pt_hs_k::run / run_hbv_stack call state.snow.distribute(parameter, false) first
    (core/pt_hs_k.h:230, core/hbv_stack.h:312; hbv_snow_common.h:44-67).  model.distribute_snow is that call for the flat state."""
    cls, par = (sb.PTHSKModel, PTHSK_DEFAULT) if stack == 1 else (sb.HbvStackModel, HBV_DEFAULT)
    m, geo, ta, st0, f = _setup(sb, cls, par, stack, n=64, T=300)
    rng = np.random.default_rng(3)
    s = st0.copy()
    s[:, 0] = rng.uniform(0.0, 300.0, 64)      # swe
    s[:, 1] = rng.uniform(0.0, 1.0, 64)        # sca
    s[:4, 0] = [0.0, 5e-4, 50.0, 50.0]         # no pack / below the 1e-3 thresholds
    s[:4, 1] = [0.5, 0.5, 0.0, 5e-4]
    s[10, 2:12] = 7.0                          # bins given: left alone
    d = m.distribute_snow(s)
    lw = par[4] if stack == 1 else par[8]
    for i in range(64):
        if i == 10:
            assert np.array_equal(d[i], s[i])
            continue
        sp, sw, swe, sca = oracle.hbv_snow_distribute(s[i, 0], s[i, 1], [1.0] * 5, [0, 0.25, 0.5, 0.75, 1.0], lw=lw)
        assert np.array_equal(d[i, 2:7], sp) and np.array_equal(d[i, 7:12], sw) and d[i, 0] == swe and d[i, 1] == sca, i
    assert np.all(d[:4, :2] == 0.0)
    # and the run from the distributed state equals the oracle's run from it (row 10's made-up bins do not match its swe: the reference
    # itself throws "Negative outflow" for such a state)
    d[10] = d[11]
    m.set_states(d)
    m.run_cells()
    run = oracle.pthsk_run_cells if stack == 1 else oracle.hbv_stack_run_cells
    want = run(geo_matrix(geo), par, f, d, ta.start * 10**6, ta.delta_t * 10**6)
    assert_parity(m.response("snow_swe"), want["snow_swe"], "snow_swe from a distributed state")
    assert_parity(m.response("avg_discharge"), want["avg_discharge"], "discharge from a distributed state")
