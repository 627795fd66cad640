"""Calibration against routed discharge (ROUTED_DISCHARGE targets, model_calibration.h:853): the single goal function against the oracle's
river routing of the oracle stack's cell discharge, and the batched form, where every member is routed through the river network with its
own cell unit hydrographs, against one-at-a-time evaluation, for pt_gs_k, pt_hs_k, hbv_stack and pt_hps_k.  Twin experiments over a snow
season on a branching network (1 -> 3 <- 2, 3 -> 4): the "observed" series is the oracle's default-parameter outflow of a river, averaged
to days."""
import os
import subprocess
import sys

import numpy as np
import pytest

from fixtures import FORCING, HBV_DEFAULT, PTGSK_DEFAULT, PTHPSK_DEFAULT, PTHSK_DEFAULT, geo_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DAY = 86400
H = 3600 * 10**6
ROUTED, DISCHARGE = 3, 0
START = 1414800000   # 2014-11-01: snow season
# stack -> (OptModel class name, default parameters, synthetic state id, oracle run, index of routing.velocity, perturbed parameters)
STACKS = {
    "pt_gs_k": ("PTGSKOptModel", PTGSK_DEFAULT, 0, "ptgsk_run_cells", 25, ((0, -3.0, -1.9), (4, -1.5, 1.0))),      # kirchner.c1, gs.tx
    "pt_hs_k": ("PTHSKOptModel", PTHSK_DEFAULT, 1, "pthsk_run_cells", 13, ((0, -3.0, -1.9), (5, -1.5, 1.5))),      # kirchner.c1, hs.tx
    "hbv_stack": ("HbvStackOptModel", HBV_DEFAULT, 2, "hbv_stack_run_cells", 17, ((0, 150.0, 450.0), (7, 0.01, 0.05))),  # soil.fc, tank.klz
    "pt_hps_k": ("PTHPSKOptModel", PTHPSK_DEFAULT, 4, "pthpsk_run_cells", 20, ((0, -3.0, -1.9), (5, -1.5, 1.5))),  # kirchner.c1, hps.tx
}
RIVERS = np.array([[1, 3, 3600.0, 1.0, 3.0, 0.0], [2, 3, 7200.0, 1.0, 5.0, 0.01], [3, 4, 10800.0, 1.0, 7.0, 0.0], [4, 0, 3600.0, 1.0, 2.0, 0.0]])
VELOCITY = 0.05   # cell distances 1 000 .. 1 775 m: unit hydrographs of 6 .. 10 hourly steps


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def _base(stack, velocity=VELOCITY):
    par = STACKS[stack][1].copy()
    par[STACKS[stack][4]] = velocity
    return par


def _perturbed(stack, rng, k, routing=False, velocity=VELOCITY):
    P = np.tile(_base(stack, velocity), (k, 1))
    for i, lo, hi in STACKS[stack][5]:
        P[:, i] = rng.uniform(lo, hi, k)
    if routing:   # velocity, alpha, beta
        off = STACKS[stack][4]
        P[:, off] = velocity * rng.uniform(0.5, 1.5, k)
        P[:, off + 1] = rng.uniform(2.0, 9.0, k)
        P[:, off + 2] = rng.uniform(0.0, 0.02, k)
    return P


def _model(sb, stack, n, T, cells_per_catchment, rivers=RIVERS, velocity=VELOCITY):
    """-> (OptModel in the default state with the river network, geo, time axis, initial state, forcing)"""
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, 9, config_index=2, cells_per_catchment=cells_per_catchment, with_routing=True, start=START)
    st0 = synthetic.default_state(STACKS[stack][2], n)
    m = getattr(sb, STACKS[stack][0])(geo, _base(stack, velocity))
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(st0)
    m.set_river_network(rivers)
    return m, geo, ta, st0


def _routed_target(sb, obs, ta, rid, scale=1.0, mode=0, **kw):
    return sb.TargetSpecification(obs, ta.start, DAY, [], scale, mode, catchment_property=ROUTED, river_id=rid, **kw)


@pytest.fixture(scope="module", params=list(STACKS))
def setup(request, sb, oracle):
    stack = request.param
    n, T = 128, 24 * 30
    m, geo, ta, st0 = _model(sb, stack, n, T, 32)
    f = {k: m.cell_forcing(k) for k in FORCING}
    gm = geo_matrix(geo)
    run = getattr(oracle, STACKS[stack][3])
    off = STACKS[stack][4]

    def routed(p, rid):
        """the oracle's daily outflow of river rid: the oracle stack's cell discharge through oracle.river_flows with p's cell UHGs"""
        q = run(gm, p, f, st0, ta.start * 10**6, H, ncore=8)["avg_discharge"]
        out = oracle.river_flows(RIVERS, rid, q, gm[:, 10].astype(np.int64), gm[:, 11], np.tile(p[off:off + 3], (n, 1)), H)[2]
        return oracle.average_to_axis(out, H, 0, 24, 30), q
    obs, q = routed(_base(stack), 4)
    return dict(stack=stack, m=m, ta=ta, gm=gm, routed=routed, obs=obs, q=q, n=n)


def _batch_equals_single(opt, P, check=None):
    batch = opt.calculate_goal_function_batch(P)
    idx = range(len(P)) if check is None else check
    single = np.array([opt.calculate_goal_function(P[i]) for i in idx])
    assert np.array_equal(batch[list(idx)], single)
    return batch


def test_single_evaluation_matches_the_oracle(sb, oracle, setup):
    c = setup
    fns = {0: oracle.nash_sutcliffe, 1: oracle.kling_gupta, 2: oracle.abs_diff_sum, 3: oracle.rmse}
    for mode, fn in fns.items():
        opt = sb.Optimizer(c["m"], [_routed_target(sb, c["obs"], c["ta"], 4, mode=mode)])
        assert opt.calculate_goal_function(_base(c["stack"])) == pytest.approx(0.0, abs=1e-9), mode   # the twin reproduces itself
        p = _perturbed(c["stack"], np.random.default_rng(mode), 1, routing=True)[0]
        got = opt.calculate_goal_function(p)
        want = fn(c["obs"], c["routed"](p, 4)[0])
        assert got == pytest.approx(want, rel=1e-9), mode


def test_batch_with_fixed_routing_parameters(sb, setup):
    c = setup
    opt = sb.Optimizer(c["m"], [_routed_target(sb, c["obs"], c["ta"], 4)])
    batch = _batch_equals_single(opt, _perturbed(c["stack"], np.random.default_rng(21), 13))
    assert np.ptp(batch) > 0.0


def test_batch_with_routing_parameters_per_member(sb, oracle, setup):
    c = setup
    opt = sb.Optimizer(c["m"], [_routed_target(sb, c["obs"], c["ta"], 4, mode=1)])
    P = _perturbed(c["stack"], np.random.default_rng(22), 11, routing=True)
    off = STACKS[c["stack"]][4]
    assert len({tuple(p[off:off + 3]) for p in P}) == len(P)   # distinct unit hydrographs per member
    batch = _batch_equals_single(opt, P)
    assert batch[5] == pytest.approx(oracle.kling_gupta(c["obs"], c["routed"](P[5], 4)[0]), rel=1e-9)


def test_batch_with_a_catchment_override_carrying_its_own_routing(sb, setup):
    """cells of catchment 2 keep the override's parameters, routing velocity / alpha / beta included, in every member"""
    c = setup
    m = c["m"]
    over = _perturbed(c["stack"], np.random.default_rng(23), 1)[0]
    off = STACKS[c["stack"]][4]
    over[off:off + 3] = (0.02, 4.0, 0.01)
    m.set_catchment_parameter(2, over)
    try:
        opt = sb.Optimizer(m, [_routed_target(sb, c["obs"], c["ta"], 4)])
        _batch_equals_single(opt, _perturbed(c["stack"], np.random.default_rng(24), 7, routing=True))
    finally:
        m.remove_catchment_parameter(2)


def test_weighted_discharge_and_routed_mix_with_missing_observations(sb, setup):
    c = setup
    ta, gm = c["ta"], c["gm"]
    obs_r = c["obs"].copy()
    obs_r[3:6] = np.nan
    sel = np.isin(gm[:, 4], [1, 2])
    obs_q = c["q"][:, sel].sum(axis=1).reshape(-1, 24).mean(axis=1)
    obs_q[20:22] = np.nan
    targets = [sb.TargetSpecification(obs_q, ta.start, DAY, [1, 2], 2.0, 0), _routed_target(sb, obs_r, ta, 3, 0.5, 1, s_a=0.5, s_b=2.0)]
    opt = sb.Optimizer(c["m"], targets)
    batch = _batch_equals_single(opt, _perturbed(c["stack"], np.random.default_rng(25), 9, routing=True))
    assert np.all(np.isfinite(batch))


def _slots(cid):
    """warp segments of equal catchment (build_slots)"""
    return sum(1 for i in range(len(cid)) if i % 32 == 0 or cid[i] != cid[i - 1])


def test_unit_hydrographs_longer_than_a_chunk(sb, setup):
    """velocity 0.008 m/s, 0.5 .. 1.5 times that per member: cell UHGs of 23 .. 124 steps.  With 12 000 members the documented sizing of goal_batch gives chunks of fewer steps
    than the H history rows carried between chunks, so the history is rebuilt from more than one earlier chunk"""
    c = setup
    stack, m, ta, gm, n = c["stack"], c["m"], c["ta"], c["gm"], c["n"]
    k = 12000
    P = _perturbed(stack, np.random.default_rng(26), k, routing=True, velocity=0.008)
    off = STACKS[stack][4]
    h = max(max(1, int(d / v / 3600.0 + 0.5)) for d in (gm[gm[:, 10] > 0, 11].min(), gm[gm[:, 10] > 0, 11].max()) for v in P[:, off]) - 1
    T, nc, n_state = ta.n, 4, m.get_states().shape[1]
    per_member = n_state * n * 8 + T * nc * 16 + 3 * len(RIVERS) * T * 8 + 2 * h * n * 8
    E = min(k, 65535, (12 << 30) // per_member)
    ps = min(T, (1 << 30) // (E * _slots(gm[:, 4]) * 16))
    if stack == "pt_gs_k":
        ps = min(ps, max(8, (4 << 30) // (E * n * 40)))
    ps = max(1, min(ps, (2 << 30) // (E * n * 16)))
    assert E == k and ps < h and T > 3 * ps, (E, ps, h)
    opt = sb.Optimizer(m, [_routed_target(sb, c["obs"], ta, 4)])
    batch = _batch_equals_single(opt, P, check=(0, 1, 4999, k - 1))
    assert np.all(np.isfinite(batch))


def test_the_batch_is_one_device_pass(sb, setup):
    c = setup
    m = c["m"]
    opt = sb.Optimizer(m, [_routed_target(sb, c["obs"], c["ta"], 4)])
    P = _perturbed(c["stack"], np.random.default_rng(3), 40, routing=True)

    def launches(fn):
        k0 = m.kernel_launches()
        fn()
        return m.kernel_launches() - k0
    d4 = launches(lambda: opt.calculate_goal_function_batch(P[:4]))
    d40 = launches(lambda: opt.calculate_goal_function_batch(P))
    d_single = launches(lambda: [opt.calculate_goal_function(p) for p in P])
    assert d4 == d40 < d_single


def test_more_sets_than_one_pass_holds(sb):
    """65 537 sets on a tiny region: grid layers are limited to 65 535 members, so the batch runs in two passes"""
    m, geo, ta, st0 = _model(sb, "hbv_stack", 64, 96, 32, rivers=np.array([[1, 2, 3600.0, 1.0, 3.0, 0.0], [2, 0, 7200.0, 1.0, 5.0, 0.0]]))
    m.run_cells()
    obs = m.river_output_flow_m3s(2).reshape(-1, 24).mean(axis=1)
    opt = sb.Optimizer(m, [_routed_target(sb, obs, ta, 2)])
    P = _perturbed("hbv_stack", np.random.default_rng(17), 65537, routing=True)
    batch = opt.calculate_goal_function_batch(P)
    for i in (0, 65534, 65535, 65536):
        assert batch[i] == opt.calculate_goal_function(P[i]), i


def test_a_batch_leaves_the_model_as_it_was(sb, setup):
    c = setup
    m = c["m"]
    opt = sb.Optimizer(m, [_routed_target(sb, c["obs"], c["ta"], 4)])
    P = _perturbed(c["stack"], np.random.default_rng(41), 5, routing=True)
    opt.calculate_goal_function(P[0])

    def snapshot():
        return (m.get_region_parameter(), m.get_states(), m.catchment_discharges(), m.river_output_flow_m3s(4), m.river_output_flow_m3s(3))
    before = snapshot()
    opt.calculate_goal_function_batch(P[1:])
    k0 = m.kernel_launches()
    m.river_output_flow_m3s(4)
    assert m.kernel_launches() == k0   # the model's routed flows are still valid: read back, not recomputed
    after = snapshot()
    for a, b in zip(before, after):
        assert np.array_equal(a, b)
    assert np.array_equal(after[0], P[0])


def test_errors_are_those_of_single_evaluation(sb, setup):
    c = setup
    m = c["m"]
    P = _perturbed(c["stack"], np.random.default_rng(43), 3, routing=True)

    def messages(opt):
        with pytest.raises(RuntimeError) as single:
            opt.calculate_goal_function(P[0])
        with pytest.raises(RuntimeError) as batch:
            opt.calculate_goal_function_batch(P)
        return str(single.value), str(batch.value)
    s, b = messages(sb.Optimizer(m, [_routed_target(sb, c["obs"], c["ta"], 99)]))
    assert s == b and "river id 99 not found" in s
    m.set_river_network(np.zeros((0, 6)))
    try:
        s, b = messages(sb.Optimizer(m, [_routed_target(sb, c["obs"], c["ta"], 4)]))
        assert s == b and "river network is empty" in s
    finally:
        m.set_river_network(RIVERS)


def test_red_zones_stay_intact_in_a_batch():
    env = dict(os.environ, SB2_GUARD="1")
    prog = f"""
import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
import numpy as np
import shyft_b200 as sb
from shyft_b200 import capi, synthetic
from fixtures import PTGSK_DEFAULT
par = PTGSK_DEFAULT.copy()
par[25] = 0.015   # cell distances up to 4 175 m: unit hydrographs of up to 97 steps with the members' velocities
n, T = 512, 24 * 20
geo, ta, env = synthetic.make_region(n, T, 9, config_index=2, cells_per_catchment=128, with_routing=True, start={START})
m = sb.PTGSKOptModel(geo, par)
m.run_interpolation(sb.InterpolationParameter(), ta, env)
m.set_states(synthetic.default_state(0, n))
m.set_river_network(np.array([[1, 3, 3600.0, 1.0, 3.0, 0.0], [2, 3, 7200.0, 1.0, 5.0, 0.0], [3, 0, 3600.0, 1.0, 2.0, 0.0], [4, 3, 0.0, 1.0, 2.0, 0.0]]))
m.run_cells()
obs = m.river_output_flow_m3s(3).reshape(-1, 24).mean(axis=1)
q = m.catchment_discharges()[:, 0].reshape(-1, 24).mean(axis=1)
opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, 86400, [], 1.0, 0, catchment_property=3, river_id=3),
                       sb.TargetSpecification(q, ta.start, 86400, [1], 1.0, 1)])
P = np.tile(par, (6, 1))
P[:, 0] = np.linspace(0.9, 1.1, 6) * par[0]
P[:, 25] = np.linspace(0.8, 1.2, 6) * par[25]
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
    """PTHSKOptimizer on a routed target: the batch equals one-at-a-time evaluation, and a population driver hands every generation to the
    device in one batch"""
    import shyft_b200 as sb
    from shyft_b200 import synthetic
    n, T = 128, 24 * 30
    geo, ta, env = synthetic.make_region(n, T, 9, config_index=2, cells_per_catchment=32, with_routing=True, start=START)
    envd = {k: getattr(env, k) for k in sb.capi.FORCING_NAMES}
    par = _base("pt_hs_k")
    m = cpp.PTHSKOptModel(geo, list(par))
    assert m.run_interpolation(ta.start * 10**6, 3600 * 10**6, T, envd)
    m.set_states(synthetic.default_state(1, n))
    m.set_river_network(RIVERS)
    m.run_cells()
    obs = np.asarray(m.river_output_flow_m3s(4)).reshape(-1, 24).mean(axis=1)
    target = cpp.TargetSpecificationPts(list(obs), ta.start * 10**6, 86400 * 10**6, [], 1.0, cpp.NASH_SUTCLIFFE,
                                        catchment_property=cpp.ROUTED_DISCHARGE, river_id=4)
    P = _perturbed("pt_hs_k", np.random.default_rng(2), 6, routing=True)
    active = (0, 13)   # kirchner.c1, routing.velocity
    lo, hi = list(par), list(par)
    for i in active:
        lo[i], hi[i] = float(P[:, i].min()), float(P[:, i].max())
    opt = cpp.PTHSKOptimizer(m, [target], lo, hi)
    assert opt.calculate_goal_function(list(par)) == pytest.approx(0.0, abs=1e-9)
    g_batch = opt.calculate_goal_function_batch(P)
    assert g_batch == [opt.calculate_goal_function(list(p)) for p in P]
    start = list(par)
    for i in active:
        start[i] = lo[i]
    b0, s0, n0 = opt.n_batch_calls, opt.n_single_calls, opt.trace_size
    best = opt.optimize_dream(start, 32)               # 8 chains: the initial population + 3 generations = 4 batches
    assert opt.n_batch_calls - b0 == 4 and opt.n_single_calls == s0 and opt.trace_size - n0 == 32
    assert opt.calculate_goal_function(best) <= opt.calculate_goal_function(start)
