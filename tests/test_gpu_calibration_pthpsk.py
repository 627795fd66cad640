"""Calibration of the pt_hps_k stack (model_calibration.h:691-699, 830-899): the single goal function against the oracle, and the batched
form, whose members are grid layers of pthpsk_run_kernel<true>, against one-at-a-time evaluation.  A twin experiment over a snow season:
the "observed" series is the oracle's default-parameter run of catchments 1 + 2, averaged to days."""
import os
import subprocess
import sys

import numpy as np
import pytest

from fixtures import FORCING, PTHPSK_DEFAULT, geo_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DAY = 86400
H = 3600 * 10**6
SID = 4   # synthetic.default_state id of pt_hps_k


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def _perturbed(rng, k):
    """k parameter sets around the default; calculate_iso_pot_energy alternates 0 / 1, so that neighbouring members of one launch take
    different branches of the snow step"""
    P = np.tile(PTHPSK_DEFAULT, (k, 1))
    P[:, 0] = rng.uniform(-3.0, -1.9, k)      # kirchner.c1
    P[:, 1] = rng.uniform(0.8, 0.99, k)       # c2
    P[:, 2] = rng.uniform(-0.15, -0.05, k)    # c3
    P[:, 3] = rng.uniform(0.5, 2.5, k)        # ae scale
    P[:, 5] = rng.uniform(-1.5, 1.5, k)       # hps.tx
    P[:, 7] = rng.uniform(1.0, 3.0, k)        # hps.wind_scale
    P[:, 12] = rng.uniform(2.0, 8.0, k)       # hps.fast_albedo_decay_rate
    P[:, 13] = rng.uniform(2.0, 8.0, k)       # hps.slow_albedo_decay_rate
    P[:, 15] = np.arange(k) % 2               # hps.calculate_iso_pot_energy
    P[:, 17] = rng.uniform(0.8, 1.4, k)       # p_corr
    return P


def _region(sb, n, T, n_stations, cells_per_catchment):
    """an OptModel of the synthetic region from 2014-11-01 (snow season), interpolated, in the default state and run once"""
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, n_stations, config_index=2, cells_per_catchment=cells_per_catchment, start=1414800000)
    m = sb.PTHPSKOptModel(geo, PTHPSK_DEFAULT)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(synthetic.default_state(SID, n))
    m.run_cells()
    return m, ta


@pytest.fixture(scope="module")
def setup(sb, oracle):
    from shyft_b200 import synthetic
    n, T = 192, 24 * 60
    geo, ta, env = synthetic.make_region(n, T, 16, config_index=2, cells_per_catchment=64, start=1414800000)  # 2014-11-01: snow season
    st0 = synthetic.default_state(SID, n)
    m = sb.PTHPSKOptModel(geo, PTHPSK_DEFAULT)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(st0)
    f = {k: m.cell_forcing(k) for k in FORCING}
    gm = geo_matrix(geo)

    def run(p):
        return oracle.pthpsk_run_cells(gm, p, f, st0, ta.start * 10**6, H, ncore=8)
    truth = run(PTHPSK_DEFAULT)
    assert truth["state"][:, 21].max() > 5.0   # snow on the ground at the end (state column 21 = swe)
    sel = np.isin(gm[:, 4], [1, 2])
    obs = oracle.average_to_axis(truth["avg_discharge"][:, sel].sum(axis=1), H, 0, 24, 60)
    return dict(m=m, run=run, ta=ta, gm=gm, sel=sel, obs=obs, truth=truth)


def _sim(oracle, c, p):
    """the oracle's daily discharge of catchments 1 + 2 under parameters p"""
    return oracle.average_to_axis(c["run"](p)["avg_discharge"][:, c["sel"]].sum(axis=1), H, 0, 24, 60)


def _batch_equals_single(opt, P):
    batch = opt.calculate_goal_function_batch(P)
    single = np.array([opt.calculate_goal_function(p) for p in P])
    assert np.array_equal(batch, single)
    return batch


def test_goal_function_matches_the_reference_formulas(sb, oracle, setup):
    c = setup
    m, ta, obs = c["m"], c["ta"], c["obs"]
    fns = {0: oracle.nash_sutcliffe, 1: oracle.kling_gupta, 2: oracle.abs_diff_sum, 3: oracle.rmse}
    for mode, fn in fns.items():
        opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, DAY, [1, 2], 1.0, mode)])
        assert opt.calculate_goal_function(PTHPSK_DEFAULT) == pytest.approx(0.0, abs=1e-9), mode  # the twin reproduces itself
        p = _perturbed(np.random.default_rng(mode), 2)[mode % 2]   # iso_pot_energy off for modes 0 and 2, on for 1 and 3
        got = opt.calculate_goal_function(p)
        want = fn(obs, _sim(oracle, c, p))
        assert got == pytest.approx(want, rel=1e-9), mode
        # the calculation filter is the union of the target catchments (prepare_optimize, :517-552): catchment 3 is not stepped
        assert np.all(m.catchment_discharges()[:, 2] == 0.0) and np.any(m.catchment_discharges()[:, 0] > 0.0)


def test_batched_ensemble_equals_one_at_a_time(sb, oracle, setup):
    c = setup
    opt = sb.Optimizer(c["m"], [sb.TargetSpecification(c["obs"], c["ta"].start, DAY, [1, 2], 1.0, 0)])
    P = _perturbed(np.random.default_rng(21), 37)
    batch = opt.calculate_goal_function_batch(P)
    single = np.array([opt.calculate_goal_function(p) for p in P])
    assert np.array_equal(batch, single)  # same arithmetic per member as the single-set kernel
    assert np.argmin(batch) == np.argmin(single) and np.ptp(batch) > 0.0
    for i in (0, 17, 36):
        assert batch[i] == pytest.approx(oracle.nash_sutcliffe(c["obs"], _sim(oracle, c, P[i])), rel=1e-9), i


def test_weighted_multi_target_batch_with_missing_observations(sb, oracle, setup):
    c = setup
    ta, gm = c["ta"], c["gm"]
    obs2 = c["obs"].copy()
    obs2[7:11] = np.nan
    sel3 = gm[:, 4] == 3
    obs3 = oracle.average_to_axis(c["truth"]["avg_discharge"][:, sel3].sum(axis=1), H, 24 * 10, 6, 100)  # 6-hourly target from day 10
    targets = [sb.TargetSpecification(obs2, ta.start, DAY, [1, 2], 2.0, 0),
               sb.TargetSpecification(obs3, ta.start + 10 * DAY, 6 * 3600, [3], 0.5, 1, s_r=1.0, s_a=0.5, s_b=2.0)]
    opt = sb.Optimizer(c["m"], targets)
    P = _perturbed(np.random.default_rng(9), 11)
    batch = _batch_equals_single(opt, P)
    q = c["run"](P[4])["avg_discharge"]
    g1 = oracle.nash_sutcliffe(obs2, oracle.average_to_axis(q[:, c["sel"]].sum(axis=1), H, 0, 24, 60))
    g2 = oracle.kling_gupta(obs3, oracle.average_to_axis(q[:, sel3].sum(axis=1), H, 240, 6, 100), 1.0, 0.5, 2.0)
    assert batch[4] == pytest.approx((2.0 * g1 + 0.5 * g2) / 2.5, rel=1e-9)


def test_cell_charge_targets_and_the_shared_series_cache(sb, oracle, setup):
    """CELL_CHARGE targets, ABS_DIFF on them scaled by max_abs_average_accessor, and the one cache vector the reference keeps for
    discharge and charge sums (the first DISCHARGE / CELL_CHARGE target decides the series every such target sees), batched"""
    c = setup
    m, ta, obs, sel = c["m"], c["ta"], c["obs"], c["sel"]
    charge_obs = oracle.average_to_axis(c["truth"]["charge_m3s"][:, sel].sum(axis=1), H, 0, 24, 60) + 0.25
    P = _perturbed(np.random.default_rng(11), 9)
    run = c["run"](P[0])
    ch, q = run["charge_m3s"][:, sel].sum(axis=1), run["avg_discharge"][:, sel].sum(axis=1)
    sim_c, scale_c = oracle.average_to_axis(ch, H, 0, 24, 60), oracle.max_abs_average_to_axis(ch, H, 0, 24, 60)
    sim_q, scale_q = oracle.average_to_axis(q, H, 0, 24, 60), oracle.max_abs_average_to_axis(q, H, 0, 24, 60)
    cases = [([sb.TargetSpecification(charge_obs, ta.start, DAY, [1, 2], 1.0, 3, catchment_property=4)], oracle.rmse(charge_obs, sim_c)),
             ([sb.TargetSpecification(charge_obs, ta.start, DAY, [1, 2], 1.0, 2, catchment_property=4)],
              oracle.abs_diff_sum_scaled(charge_obs, sim_c, scale_c)),
             ([sb.TargetSpecification(obs, ta.start, DAY, [1, 2], 1.0, 0),
               sb.TargetSpecification(charge_obs, ta.start, DAY, [1, 2], 3.0, 2, catchment_property=4)],
              (oracle.nash_sutcliffe(obs, sim_q) + 3.0 * oracle.abs_diff_sum_scaled(charge_obs, sim_q, scale_q)) / 4.0),
             ([sb.TargetSpecification(charge_obs, ta.start, DAY, [1, 2], 3.0, 3, catchment_property=4),
               sb.TargetSpecification(obs, ta.start, DAY, [1, 2], 1.0, 0)],
              (3.0 * oracle.rmse(charge_obs, sim_c) + oracle.nash_sutcliffe(obs, sim_c)) / 4.0)]
    for k, (targets, want) in enumerate(cases):
        batch = _batch_equals_single(sb.Optimizer(m, targets), P)
        assert batch[0] == pytest.approx(want, rel=1e-9), k


def test_the_batch_is_one_device_pass(sb, setup):
    """launches of a batch do not grow with the number of sets: one step launch, one catchment reduction and one goal kernel"""
    c = setup
    m = c["m"]
    opt = sb.Optimizer(m, [sb.TargetSpecification(c["obs"], c["ta"].start, DAY, [1, 2], 1.0, 0)])
    P = _perturbed(np.random.default_rng(3), 40)

    def launches(fn):
        k0 = m.kernel_launches()
        fn()
        return m.kernel_launches() - k0
    d4 = launches(lambda: opt.calculate_goal_function_batch(P[:4]))
    d40 = launches(lambda: opt.calculate_goal_function_batch(P))
    d_single = launches(lambda: [opt.calculate_goal_function(p) for p in P])
    assert d4 == d40 == 3
    assert d40 < d_single


def test_time_split_on_and_off(sb):
    """members are time-sliced while (cell groups x members) < 16 000 and stepped whole-chunk beyond: both equal single evaluation
    (which slices: 63 cell groups)"""
    m, ta = _region(sb, 2000, 24 * 20, 16, 700)
    obs = m.catchment_discharges()[:, :2].sum(axis=1).reshape(-1, 24).mean(axis=1)
    opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, DAY, [1, 2], 1.0, 0)])
    P = _perturbed(np.random.default_rng(13), 256)   # 63 groups x 256 members = 16 128: no time split
    one = opt.calculate_goal_function_batch(P[:1])   # 63 groups x 1 member: time split
    assert one[0] == opt.calculate_goal_function(P[0])
    batch = opt.calculate_goal_function_batch(P)
    assert batch[0] == one[0]
    for i in (0, 101, 255):
        assert batch[i] == opt.calculate_goal_function(P[i]), i


def test_more_sets_than_one_pass_holds(sb):
    """65 537 sets: grid layers are limited to 65 535 members, so the batch runs in two passes"""
    m, ta = _region(sb, 64, 96, 4, 32)
    obs = m.catchment_discharges()[:, 0].reshape(-1, 24).mean(axis=1)
    opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, DAY, [1], 1.0, 0)])
    P = _perturbed(np.random.default_rng(17), 65537)
    k0 = m.kernel_launches()
    batch = opt.calculate_goal_function_batch(P)
    assert m.kernel_launches() - k0 == 2 * 3   # two passes of (step, catchment reduction, goal)
    for i in (0, 65534, 65535, 65536):
        assert batch[i] == opt.calculate_goal_function(P[i]), i


def test_targets_without_a_device_batch_go_one_set_at_a_time(sb, oracle, setup):
    """a target axis shifted by half a step, and a snow water equivalent target, are evaluated set by set"""
    c = setup
    m, ta = c["m"], c["ta"]
    P = _perturbed(np.random.default_rng(31), 3)
    opt = sb.Optimizer(m, [sb.TargetSpecification(c["obs"][:59], ta.start + 1800, DAY, [1, 2], 1.0, 3)])
    k0 = m.kernel_launches()
    batch = opt.calculate_goal_function_batch(P)
    k1 = m.kernel_launches()
    assert np.array_equal(batch, [opt.calculate_goal_function(p) for p in P])
    assert k1 - k0 == m.kernel_launches() - k1   # the batch is the loop over the single entry
    sel, area = c["sel"], c["gm"][:, 3]
    swe_obs = oracle.average_to_axis((c["truth"]["snow_swe"][:, sel] * area[sel]).sum(axis=1) / area[sel].sum(), H, 0, 24, 60)
    opt = sb.Optimizer(m, [sb.TargetSpecification(swe_obs, ta.start, DAY, [1, 2], 1.0, 3, catchment_property=2)])
    k0 = m.kernel_launches()
    batch = opt.calculate_goal_function_batch(P)
    k1 = m.kernel_launches()
    assert np.array_equal(batch, [opt.calculate_goal_function(p) for p in P])
    assert k1 - k0 == m.kernel_launches() - k1
    run = c["run"](P[1])
    sim = oracle.average_to_axis((run["snow_swe"][:, sel] * area[sel]).sum(axis=1) / area[sel].sum(), H, 0, 24, 60)
    assert batch[1] == pytest.approx(oracle.rmse(swe_obs, sim), rel=1e-9)


def test_a_batch_leaves_the_model_as_it_was(sb, setup):
    c = setup
    m = c["m"]
    opt = sb.Optimizer(m, [sb.TargetSpecification(c["obs"], c["ta"].start, DAY, [1, 2], 1.0, 0)])
    P = _perturbed(np.random.default_rng(41), 5)
    opt.calculate_goal_function(P[0])
    before = (m.get_region_parameter(), m.get_states(), m.catchment_discharges())
    opt.calculate_goal_function_batch(P[1:])
    after = (m.get_region_parameter(), m.get_states(), m.catchment_discharges())
    for a, b in zip(before, after):
        assert np.array_equal(a, b)
    assert np.array_equal(after[0], P[0])


def test_a_catchment_override_outside_the_targets(sb, setup):
    """cells under a catchment parameter keep it in every member (model_calibration.h:830-832)"""
    c = setup
    m = c["m"]
    m.set_catchment_parameter(3, _perturbed(np.random.default_rng(51), 2)[1])
    try:
        opt = sb.Optimizer(m, [sb.TargetSpecification(c["obs"], c["ta"].start, DAY, [1, 2], 1.0, 0)])
        _batch_equals_single(opt, _perturbed(np.random.default_rng(52), 7))
    finally:
        m.remove_catchment_parameter(3)


def test_red_zones_stay_intact_in_a_batch():
    env = dict(os.environ, SB2_GUARD="1")
    prog = f"""
import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
import numpy as np
import shyft_b200 as sb
from shyft_b200 import capi, synthetic
from fixtures import PTHPSK_DEFAULT as par
n, T = 2000, 24 * 20
geo, ta, env = synthetic.make_region(n, T, 9, config_index=2, cells_per_catchment=500, start=1414800000)
m = sb.PTHPSKOptModel(geo, par)
m.run_interpolation(sb.InterpolationParameter(), ta, env)
m.set_states(synthetic.default_state({SID}, n))
m.run_cells()
obs = m.catchment_discharges()[:, :2].sum(axis=1).reshape(-1, 24).mean(axis=1)
opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, 86400, [1, 2], 1.0, 0),
                       sb.TargetSpecification(obs, ta.start, 86400, [1, 2], 1.0, 2, catchment_property=4)])
P = np.tile(par, (6, 1))
P[:, 0] = np.linspace(0.9, 1.1, 6) * par[0]
P[:, 15] = np.arange(6) % 2
g = opt.calculate_goal_function_batch(P)
assert np.all(np.isfinite(g)) and g[0] == opt.calculate_goal_function(P[0])
v, msg = capi.check_guards()
print('batch ok', g.tolist(), 'guards', v, msg)
sys.exit(1 if v else 0)
"""
    r = subprocess.run([sys.executable, "-c", prog], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "batch ok" in r.stdout and "guards 0" in r.stdout


@pytest.fixture(scope="module")
def cpp():
    from shyft_b200 import _build
    _build.build_pybind_module()
    from shyft_b200 import _shyft_b200_cpp
    return _shyft_b200_cpp


def test_optimizer_through_the_module(cpp):
    """PTHPSKOptimizer: the batch equals one-at-a-time evaluation, and a population driver hands every generation to the device in one
    batch"""
    import shyft_b200 as sb
    from shyft_b200 import synthetic
    n, T = 192, 24 * 60
    geo, ta, env = synthetic.make_region(n, T, 16, config_index=2, cells_per_catchment=64, start=1414800000)
    envd = {k: getattr(env, k) for k in sb.capi.FORCING_NAMES}
    par, active = PTHPSK_DEFAULT, (0, 5)   # kirchner.c1, hps.tx
    m = cpp.PTHPSKOptModel(geo, list(par))
    assert m.run_interpolation(ta.start * 10**6, 3600 * 10**6, T, envd)
    m.set_states(synthetic.default_state(SID, n))
    m.run_cells()
    q = m.catchment_discharges()                      # [catchment][step]
    obs_daily = (q[0] + q[1]).reshape(-1, 24).mean(axis=1)
    target = cpp.TargetSpecificationPts(list(obs_daily), ta.start * 10**6, 86400 * 10**6, [1, 2], 1.0, cpp.NASH_SUTCLIFFE)
    P = _perturbed(np.random.default_rng(2), 6)
    lo, hi = list(par), list(par)
    for i in active:
        lo[i], hi[i] = float(P[:, i].min()), float(P[:, i].max())
    opt = cpp.PTHPSKOptimizer(m, [target], lo, hi)
    assert [i for i in range(len(par)) if opt.parameter_active(i)] == list(active)
    assert opt.calculate_goal_function(list(par)) == pytest.approx(0.0, abs=1e-9)      # the twin reproduces itself
    g_batch = opt.calculate_goal_function_batch(P)
    g_single = [opt.calculate_goal_function(list(p)) for p in P]
    assert g_batch == g_single
    start = list(par)
    for i in active:
        start[i] = lo[i]
    b0, s0, n0 = opt.n_batch_calls, opt.n_single_calls, opt.trace_size
    best = opt.optimize_dream(start, 32)               # 8 chains: the initial population + 3 generations = 4 batches
    assert opt.n_batch_calls - b0 == 4 and opt.n_single_calls == s0 and opt.trace_size - n0 == 32
    assert opt.calculate_goal_function(best) <= opt.calculate_goal_function(start)
