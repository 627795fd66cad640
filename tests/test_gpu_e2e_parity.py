"""End-to-end parity of the SHIPPED path -- sb2_run_windowed: dense DMMA interpolation (BTK temperature + IDW) feeding the step kernels
window by window, exactly what bench.py times -- against the oracle's interpolate -> run_cells on the same inputs, with a census of the
discrete decisions that flipped (tests/e2e_census.py).  core/region_model.h:397-527 -> :578-597; BASELINE.md section 5.

What is asserted:
  * the interpolated forcing is within 1e-11 of the oracle's everywhere (it differs: the tensor-core contraction sums in another order);
  * every cell-step of every cell WITHOUT a decision flip is within the contractual 1e-9 (by construction of the census) and the share
    of cell-steps within 1e-9 stays above a committed bound;
  * every first divergence is attributed to a known decision (Brent's search in corr_lwc, precipitation phase, sign of T, the
    Priestley-Taylor cancellation next to zero, Runge-Kutta accept / reject) -- nothing "unattributed";
  * the flip rate is of the size the REFERENCE ALGORITHM shows under a 1e-13 forcing perturbation on the CPU (tests/test_e2e_census_cpu.py).
The census of each run is written to e2e_census_<stack>.json in the test's temporary directory (bench.py reports its own, smaller one).
"""
import json
import os

import numpy as np
import pytest

from e2e_cases import oracle_forcing, region_slice, run_device_windows
from e2e_census import Census
from fixtures import HBV_DEFAULT, PTGSK_DEFAULT, PTHPSK_DEFAULT, PTHSK_DEFAULT, PTSSK_DEFAULT, geo_matrix
from parity import assert_parity

pytestmark = pytest.mark.gpu
KNOWN_CAUSES = {"brent_corr_lwc", "precipitation_phase_T_lt_tx", "sign_of_T", "pe_cancellation_next_to_zero", "rk_accept_reject"}


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def _save(d, name, c):
    with open(os.path.join(d, f"e2e_census_{name}.json"), "w") as f:
        json.dump(c, f, indent=1)


def test_config2_slice_pt_gs_k_windowed_dense_interpolation_census(sb, oracle, tmp_path):
    """BASELINE configs[1]: 2 048 cells (128 runs of 16 neighbours spread over the 100 000-cell region) x 2 years, 64 stations,
    BTK temperature + IDW, windows of 2 048 steps, dense DMMA interpolation on (the default)."""
    from shyft_b200 import synthetic
    T, W = 17520, 2048
    geo, ta, env = region_slice(100000, T, 64, 128, config_index=1)
    n = geo.shape[0]
    st0 = synthetic.default_state(0, n)
    gm, f = oracle_forcing(oracle, geo, ta, env, btk_temperature=True)
    want = oracle.ptgsk_run_cells(gm, PTGSK_DEFAULT, f, st0, ta.start * 10**6, ta.delta_t * 10**6, collect_response=True, collect_state=True, ncore=16)
    assert np.nanmax(want["snow_swe"]) > 10.0, "the slice must build a snow pack"
    end_state = want.pop("state")

    m = sb.PTGSKModel(geo, PTGSK_DEFAULT)
    m.set_state_collection(-1, True)
    m.initialize_cell_environment(ta)
    m._set_sources(env)
    m.set_states(st0)
    ip = sb.InterpolationParameter()   # BTK temperature + IDW, the defaults of core/region_model.h:65-95
    cs = Census(want, f, tx=PTGSK_DEFAULT[4])
    resp = ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output")
    run_device_windows(m, ip, T, W, resp, sb.capi.STATE_SERIES_NAMES[sb.PT_GS_K], cs.add_window)
    c = cs.result()
    cq_chunked = m.catchment_discharges()
    _save(tmp_path, "pt_gs_k", c)
    print("e2e census pt_gs_k:", json.dumps({k: c[k] for k in ("cell_steps_within", "cells_with_a_decision_flip", "flip_rate_per_cell_year",
                                                                 "first_divergence_by_cause", "forcing_worst_rel")}))
    assert all(v == 0 for v in c["forcing_outside_1e-11"].values()), c["forcing_outside_1e-11"]
    assert set(c["first_divergence_by_cause"]) <= KNOWN_CAUSES, c["first_divergence_by_cause"]
    # committed bounds (DESIGN.md section 2): measured 0.98 / 0.04 flips per cell-year on the B200; the CPU oracle under a 1e-13
    # forcing perturbation shows the same (tests/test_e2e_census_cpu.py)
    assert c["cell_steps_within"] >= 0.95, c["cell_steps_within"]
    assert c["flip_rate_per_cell_year"] <= 0.10, c["flip_rate_per_cell_year"]
    for k in ("gs_albedo", "gs_surface_heat", "gs_alpha", "gs_sdc_melt_mean", "gs_acc_melt", "gs_temp_swe"):
        assert c["series"][k]["outside"] == 0, (k, c["series"][k])   # the decisions that flip touch liquid water only
    # cells without a flip: end state within 1e-9 as well
    flipped = np.zeros(n, dtype=bool)
    for k in cs.names:
        flipped |= cs.bad[k].any(axis=0)
    assert_parity(m.get_states()[~flipped], end_state[~flipped], "end state of the cells without a flip")
    # the same run as ONE call over the whole axis (what bench.py does): catchment sums bit-identical to the window-by-window drive
    m.revert_to_initial_state()
    m.run_windowed(ip, window_steps=W)
    assert np.array_equal(m.catchment_discharges(), cq_chunked)


@pytest.mark.parametrize("stack", ["pt_hs_k", "hbv_stack", "pt_ss_k", "pt_hps_k"])
def test_config3_slice_hbv_windowed_with_routing_census(sb, oracle, stack, tmp_path):
    """BASELINE configs[2] shape: 1 024 cells cut out of the 400 000-cell grid x 1 year from November, river network routing."""
    from shyft_b200 import synthetic
    T, W = 8760, 1024
    geo, ta, env = region_slice(400000, T, 64, 64, config_index=2, with_routing=True, start=1414800000)
    n = geo.shape[0]
    cls, par, sid, run = {"pt_hs_k": (sb.PTHSKModel, PTHSK_DEFAULT, 1, oracle.pthsk_run_cells),
                          "hbv_stack": (sb.HbvStackModel, HBV_DEFAULT, 2, oracle.hbv_stack_run_cells),
                          "pt_ss_k": (sb.PTSSKModel, PTSSK_DEFAULT, 3, oracle.ptssk_run_cells),
                          "pt_hps_k": (sb.PTHPSKModel, PTHPSK_DEFAULT, 4, oracle.pthpsk_run_cells)}[stack]
    st0 = synthetic.default_state(sid, n)
    gm, f = oracle_forcing(oracle, geo, ta, env, btk_temperature=True)
    want = run(gm, par, f, st0, ta.start * 10**6, ta.delta_t * 10**6, ncore=16)
    end_state = want.pop("state")
    m = cls(geo, par)
    m.initialize_cell_environment(ta)
    m._set_sources(env)
    m.set_states(st0)
    ip = sb.InterpolationParameter()
    cs = Census(want, f, tx=0.0, watch=())
    q_dev = np.zeros((T, n))

    def on_window(w0, got, fg):
        q_dev[w0:w0 + got["avg_discharge"].shape[0]] = got["avg_discharge"]
        cs.add_window(w0, got, fg)
    if stack != "hbv_stack":
        want.pop("soil_outflow", None)   # hbv_stack only
    run_device_windows(m, ip, T, W, [k for k in want if want[k].shape == (T, n)], (), on_window)
    c = cs.result()
    _save(tmp_path, stack, c)
    print(f"e2e census {stack}:", json.dumps({k: c[k] for k in ("cell_steps_within", "cells_with_a_decision_flip", "first_divergence_by_cause",
                                                                  "forcing_worst_rel")}))
    assert all(v == 0 for v in c["forcing_outside_1e-11"].values()), c["forcing_outside_1e-11"]
    assert set(c["first_divergence_by_cause"]) <= KNOWN_CAUSES | {"snow_threshold_other"}, c["first_divergence_by_cause"]
    assert c["cell_steps_within"] >= 0.98, c["cell_steps_within"]
    flipped = np.zeros(n, dtype=bool)
    for k in cs.names:
        flipped |= cs.bad[k].any(axis=0)
    assert_parity(m.get_states()[~flipped], end_state[~flipped], "end state of the cells without a flip")
    # routing in one windowed pass over the whole axis (cell discharge convolved window by window, history carried over) against the
    # oracle's river network fed with the DEVICE's cell discharge: isolates routing from the decision flips above
    cids = np.unique(geo["catchment_id"])
    rivers = np.array([[cid, (cids[k + 1] if (k % 4) != 3 and k + 1 < cids.size else 0), 3600.0 * (1 + k % 4), 1.0, 7.0, 0.0] for k, cid in enumerate(cids)],
                      dtype=np.float64)
    m.set_river_network(rivers)
    m.revert_to_initial_state()
    m.run_windowed(ip, window_steps=W)
    uhg = np.tile({"pt_hs_k": par[13:16], "hbv_stack": par[17:20], "pt_ss_k": par[16:19], "pt_hps_k": par[20:23]}[stack], (n, 1))
    for rid in (cids[0], cids[3], cids[-1]):
        local, up, out = oracle.river_flows(rivers, int(rid), q_dev, gm[:, 10].astype(np.int64), gm[:, 11], uhg, ta.delta_t * 10**6)
        assert_parity(m.river_local_inflow_m3s(int(rid)), local, f"river {rid} local inflow", rtol=1e-9)
        assert_parity(m.river_output_flow_m3s(int(rid)), out, f"river {rid} output", rtol=1e-9)
