"""GPU parity of the pt_hps_k stack (core/pt_hps_k.h:201-303; hbv_physical_snow core/hbv_physical_snow.h:266-529) through the C ABI: the snow
routine one step at a time against the oracle (the reference unit-tests it the same way, test/hbv_physical_snow_test.cpp), the stack over a
winter, the reference's own stack-level asserts (test/pt_hps_k_test.cpp:97-156) on the device."""
import numpy as np
import pytest

import stack_cases as sc
from fixtures import FORCING, PTHPSK_DEFAULT, geo_matrix
from parity import assert_parity

pytestmark = pytest.mark.gpu
PAR11 = np.array([0.0, 0.1, 0.5, 2.0, 1.0, 30.0, 0.9, 0.6, 5.0, 5.0, 5.0])   # oracle.HPS_DEFAULT order


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def _bits_equal(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.array_equal(a.view(np.uint64), b.view(np.uint64)) or np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("iso", [False, True])
def test_hps_step_sequences_are_bit_identical(sb, oracle, iso):
    """hbv_physical_snow::calculator::step chained over random weather for many cells, device step by step against the oracle: pack reset,
    snowfall with bin redistribution, albedo decay, refreeze, partial and complete melt of bins, rain on snow; 1 h and 3 h steps"""
    rng = np.random.default_rng(41 + int(iso))
    n_cells, n_steps = 96, 300
    st = np.tile(np.array([0.0] * 10 + [0.4] * 5 + [0.0] * 5 + [30000.0, 0.0, 0.0]), (n_cells, 1))
    st_o = st.copy()
    season = np.sin(2 * np.pi * np.arange(n_steps) / n_steps)
    bad_seen = 0
    saw_pack = False
    for i in range(n_steps):
        temp = -5.0 * season[i] + rng.normal(0, 4.0, n_cells)
        prec = rng.exponential(1.5, n_cells) * (rng.random(n_cells) < 0.3)
        rad = rng.uniform(0.0, 400.0, n_cells)
        wind = np.abs(rng.normal(3.0, 2.0, n_cells))
        rh = rng.uniform(0.4, 1.0, n_cells)
        dt_h = 3.0 if i % 4 == 0 else 1.0
        rows = np.concatenate([np.tile(PAR11, (n_cells, 1)), np.full((n_cells, 1), float(iso)), st, np.full((n_cells, 1), dt_h), temp[:, None],
                               rad[:, None], prec[:, None], wind[:, None], rh[:, None]], axis=1)
        got = sb.capi.unit_eval("hps_step", rows)
        for c in range(n_cells):
            try:
                s1, r = oracle.hps_step(st_o[c], temp[c], rad[c], prec[c], wind[c], rh[c], dt_us=int(dt_h * 3600 * 10**6), par=PAR11, iso=iso)
            except RuntimeError:
                assert got[c, 26] == 1.0            # the device raised its flag where the reference throws "Negative outflow"
                bad_seen += 1
                s1 = got[c, :23].copy()
            else:
                assert got[c, 26] == 0.0
                assert _bits_equal(got[c, :23], s1) and _bits_equal(got[c, 23:26], r), (i, c, got[c], s1, r)
            st_o[c] = s1
        st = got[:, :23].copy()
        saw_pack = saw_pack or st[:, 21].max() > 5.0
    assert saw_pack and bad_seen < n_cells * n_steps * 0.01


def test_hps_mass_balance_cases_on_the_device(sb, oracle):
    """test/hbv_physical_snow_test.cpp:29-176 on the device (bins from state.distribute(p), taken from the oracle)"""
    for T, prec, swe, sca in [(1.0, 0.04, 0.05, 1.0), (-1.0, 0.15, 0.2, 0.6), (0.0, 0.15, 0.2, 0.6), (0.0, 0.15, 0.0, 0.0), (3.0, 0.0, 10.0, 0.5)]:
        sp, sw, swe_d, sca_d = oracle.hbv_snow_distribute(swe, sca, [1.0] * 5, [0.0, 0.25, 0.5, 0.75, 1.0], lw=0.1)
        st = np.concatenate([sp, sw, [0.6] * 5, [1752.56396484375] * 5, [0.0, swe_d, sca_d]])
        row = np.concatenate([PAR11, [0.0], st, [1.0, T, 10.0, prec, 2.0, 0.70]])
        got = sb.capi.unit_eval("hps_step", row[None, :])[0]
        assert got[26] == 0.0
        assert got[21] + got[23] == pytest.approx(prec + swe_d, abs=1e-8)
        want, r = oracle.hps_step(st, T, 10.0, prec, 2.0, 0.70)
        assert _bits_equal(got[:23], want) and _bits_equal(got[23:26], r)


def test_pt_hps_k_stack_parity_through_a_winter(sb, oracle):
    from shyft_b200 import synthetic
    n, T = 320, 6000
    geo, ta, env = synthetic.make_region(n, T, 16, config_index=2, cells_per_catchment=40, start=1414800000)   # 2014-11-01
    m = sb.PTHPSKModel(geo, PTHPSK_DEFAULT)
    assert m.parameter_size == 24 and m.state_size == 24
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    st0 = synthetic.default_state(4, n)
    m.set_states(st0)
    m.set_state_collection(-1, True)
    f = {k: m.cell_forcing(k) for k in FORCING}
    m.run_cells()
    want = oracle.pthpsk_run_cells(geo_matrix(geo), PTHPSK_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, ncore=8)
    assert np.nanmax(want["snow_swe"]) > 5.0, "the fixture must build a snow pack"
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert_parity(m.response(name), want[name], "pt_hps_k " + name)
    assert_parity(m.get_states(), want["state"], "pt_hps_k end state")
    for name in ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output"):
        assert np.array_equal(m.response(name), want[name], equal_nan=True), "pt_hps_k " + name + " is within 1e-9 but not bit-identical"
    assert np.array_equal(m.get_states(), want["state"])
    # state series: T + 1 instant values; the first row is the initial state, the last the end state (swe over the cell, the rest as stored)
    s_end = m.get_states()
    frac = 1.0 - geo["lake"] - geo["reservoir"]
    names = sb.capi.STATE_SERIES_NAMES[sb.PT_HPS_K]
    assert len(names) == 24
    assert np.array_equal(m.state_series("snow_swe")[T], s_end[:, 21] * frac) and np.array_equal(m.state_series("snow_swe")[0], st0[:, 21] * frac)
    assert np.array_equal(m.state_series("snow_sca")[T], s_end[:, 22]) and np.array_equal(m.state_series("snow_surface_heat")[T], s_end[:, 20])
    for i in range(5):
        assert np.array_equal(m.state_series(f"snow_sp_{i}")[T], s_end[:, i]) and np.array_equal(m.state_series(f"snow_sw_{i}")[T], s_end[:, 5 + i])
        assert np.array_equal(m.state_series(f"snow_albedo_{i}")[T], s_end[:, 10 + i])
        assert np.array_equal(m.state_series(f"snow_iso_pot_energy_{i}")[T], s_end[:, 15 + i])
    assert np.array_equal(m.state_series("kirchner_discharge")[T], s_end[:, 23] * geo["area"] * (1 / (3600.0 * 1000.0))) or \
        np.allclose(m.state_series("kirchner_discharge")[T], s_end[:, 23] * geo["area"] / 3.6e6, rtol=1e-15)
    # the response snow_swe of step i is the state collector's value at i + 1
    assert np.array_equal(m.state_series("snow_swe")[1:], m.response("snow_swe"))
    cd = m.catchment_discharges()
    assert_parity(cd[:, 0], want["avg_discharge"][:, :40].sum(axis=1), "catchment discharge", rtol=1e-12)
    # chunked run = one shot; windowed run = resident run
    q, s = m.response("avg_discharge"), m.get_states()
    m.revert_to_initial_state()
    for k in range(4):
        m.run_cells(0, 1500 * k, 1500)
    assert np.array_equal(m.response("avg_discharge"), q) and np.array_equal(m.get_states(), s)
    b = sb.PTHPSKOptModel(geo, PTHPSK_DEFAULT)
    b.initialize_cell_environment(ta)
    b.set_states(st0)
    b.run_windowed(sb.InterpolationParameter(), env=env, window_steps=777)
    assert np.array_equal(b.catchment_discharges(), cd) and np.array_equal(b.get_states(), s)


def test_pt_hps_k_iso_pot_energy_and_catchment_override(sb, oracle):
    """calculate_iso_pot_energy on (the only branch that writes iso_pot_energy) in one catchment's parameter override"""
    from shyft_b200 import synthetic
    n, T = 96, 1500
    geo, ta, env = synthetic.make_region(n, T, 9, config_index=3, cells_per_catchment=32, start=1417392000)
    m = sb.PTHPSKModel(geo, PTHPSK_DEFAULT)
    over = PTHPSK_DEFAULT.copy()
    over[15] = 1.0
    over[5] = 0.5        # tx
    m.set_catchment_parameter(2, over)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    st0 = synthetic.default_state(4, n)
    m.set_states(st0)
    f = {k: m.cell_forcing(k) for k in FORCING}
    m.run_cells()
    pset = (np.asarray(geo["catchment_id"]) == 2).astype(np.int32)
    want = oracle.pthpsk_run_cells(geo_matrix(geo), np.stack([PTHPSK_DEFAULT, over]), f, st0, ta.start * 10**6, ta.delta_t * 10**6, pset_of_cell=pset, ncore=8)
    assert_parity(m.response("avg_discharge"), want["avg_discharge"], "pt_hps_k discharge with override")
    assert_parity(m.get_states(), want["state"], "pt_hps_k end state with override")
    s = m.get_states()
    assert np.any(s[pset == 1, 15:20] != 0.0) and np.all(s[pset == 0, 15:20] == 0.0)


def test_pt_hps_k_reference_known_answers_on_the_device(sb):
    """test/pt_hps_k_test.cpp:97-156 (lake / reservoir response) with the reference's own asserts (tests/stack_cases.py)"""
    models = {}

    def run(stack, geo, par, forcing, state, t0_us, T):
        assert stack == 4
        key = (geo.tobytes(), T)
        if key not in models:
            g = geo[0]
            cells = sb.geo_cell_data_vector([g[0]], [g[1]], [g[2]], area=g[3], catchment_id=np.array([int(g[4])]), radiation_slope_factor=g[5],
                                            glacier=g[6], lake=g[7], reservoir=g[8], forest=g[9])
            m = sb.PTHPSKModel(cells, par)
            m.initialize_cell_environment(sb.TimeAxis(t0_us // 10**6, 3600, T))
            m.set_state_collection(-1, True)
            models[key] = m
        m = models[key]
        m.set_region_parameter(par)
        for k in FORCING:
            m.set_cell_forcing(k, forcing[k])
        m.set_states(state)
        m.run_cells()
        out = {name: m.response(name) for name in ("avg_discharge", "snow_swe", "snow_sca", "snow_outflow")}
        out["state_snow_swe"] = m.state_series("snow_swe")
        out["state"] = m.get_states()
        return out
    sc.pthpsk_lake_reservoir_response(run)


def test_pt_hps_k_through_the_pybind_module_and_routing(sb):
    from shyft_b200 import _build, synthetic
    _build.build_pybind_module()
    from shyft_b200 import _shyft_b200_cpp as cpp
    n, T = 64, 240
    geo, ta, env = synthetic.make_region(n, T, 9, config_index=2, cells_per_catchment=32, start=1417392000, with_routing=True)
    a = cpp.PTHPSKModel(geo, list(PTHPSK_DEFAULT))
    envd = {k: getattr(env, k) for k in sb.capi.FORCING_NAMES}
    assert a.run_interpolation(ta.start * 10**6, 3600 * 10**6, T, envd)
    a.set_states(synthetic.default_state(4, n))
    a.run_cells()
    b = sb.PTHPSKModel(geo, PTHPSK_DEFAULT)
    b.run_interpolation(sb.InterpolationParameter(), ta, env)
    b.set_states(synthetic.default_state(4, n))
    b.set_state_collection(-1, True)
    b.run_cells()
    assert np.array_equal(a.catchment_discharges()[0], b.catchment_discharges()[:, 0])
    assert np.allclose(b.statistics.discharge([1]), b.response("avg_discharge")[:, :32].sum(axis=1), rtol=1e-12)
    assert b.kirchner_state.discharge([1]).shape == (T + 1,)
    # routing reads velocity / alpha / beta at offset 20 of the parameter vector
    b.set_river_network(synthetic.river_chain(2, depth=2))
    out = b.river_output_flow_m3s(2)
    assert out.shape == (T,) and np.all(np.isfinite(out)) and out.sum() > 0.0
