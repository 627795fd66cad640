"""Forcing ensembles (sb2_run_ensemble, DESIGN.md section 3.7): every member of run_ensemble against the member loop it replaces -- set
the member's sources, interpolate(best_effort=False), run_cells from the same state, read the catchment sums -- with np.array_equal, on
all five stacks; windows, ranges, overrides and the filter, sources on a point axis, passes, launches, the oracle, the model left as it
was, errors, red zones and the bindings."""
import os
import subprocess
import sys

import numpy as np
import pytest

import ensemble_cases as ec
import step_cases as sc
from test_gpu_step_paths import launched

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WINTER = 1424476800   # 2015-02-21: snowfall and a snow pack from the first step
SUMMER = 1435708800   # 2015-07-01
NAMES = ("temperature", "precipitation", "radiation", "wind_speed", "rel_hum")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def three_hourly(sb, src, ta, point_fx="average"):
    """a (xyz, values [T][S]) source as a GeoPointSources on a 3-hourly axis, with a last point at the axis end (linear between points
    leaves the steps after the last point NaN)"""
    xyz, v = src
    times = ta.start + ta.delta_t * np.arange(0, ta.n + 1, 3)
    values = np.vstack([v[::3], v[-1:]])[:times.size]
    return sb.GeoPointSources(xyz, times, values, t_end=ta.start + ta.delta_t * ta.n, point_fx=point_fx)


def case(sb, stack, n=203, days=30, E=6, stations=9, seed=0, nan=True, radiation_axis=True, cfg=3, start=WINTER):
    """-> (model with its own sources set and a state, base env, member envs, ip).  Temperature and precipitation per member; one
    member with a NaN stretch in a temperature station (BTK segments), one in a precipitation station (sparse IDW)."""
    from shyft_b200 import synthetic
    T = 24 * days
    geo, ta, env = synthetic.make_region(n, T, stations, config_index=cfg, cells_per_catchment=(n + 2) // 3, start=start)
    m = getattr(sb, sc.MODEL[stack])(geo, sc.DEFAULT[stack])
    m.initialize_cell_environment(ta)
    base = sb.RegionEnvironment(**{k: getattr(env, k) for k in NAMES})
    if radiation_axis:
        base.radiation = three_hourly(sb, env.radiation, ta)
    m._set_sources(base)
    m.set_states(synthetic.default_state(sc.STACK_ID[stack], n))
    rng = np.random.default_rng(seed)
    members = []
    for e in range(E):
        xt, vt = env.temperature
        xp, vp = env.precipitation
        vt = vt + rng.normal(0.0, 1.5, size=(1, vt.shape[1])) + rng.normal(0.0, 0.3, size=vt.shape)
        vp = vp * rng.uniform(0.5, 1.5, size=(1, vp.shape[1]))
        if nan and e == 1:
            vt = vt.copy(); vt[100:160, 2] = np.nan
        if nan and e == 2:
            vp = vp.copy(); vp[200:260, 3] = np.nan
        members.append(sb.RegionEnvironment(temperature=(xt, vt), precipitation=(xp, vp)))
    return m, base, members, sb.InterpolationParameter()


def member_loop(sb, m, base, members, ip, start_step=0, n_steps=0):
    """what run_ensemble replaces, member by member through the public single path"""
    st = m.get_states()
    first, count = (start_step, n_steps) if n_steps > 0 else (0, m.time_axis.n)
    q, c = [], []
    for env in members:
        full = sb.RegionEnvironment(**{k: getattr(env, k) if getattr(env, k) is not None else getattr(base, k) for k in NAMES})
        m.interpolate(ip, full, best_effort=False)
        m.set_states(st)
        m.run_cells(0, start_step, n_steps)
        q.append(m.catchment_discharges(first, count))
        c.append(m.catchment_charges(first, count))
    m.set_states(st)
    return np.array(q), np.array(c)


@pytest.mark.parametrize("stack", sc.STACKS)
def test_every_member_equals_the_member_loop(sb, stack):
    m, base, members, ip = case(sb, stack)
    q, c = m.run_ensemble(ip, members)
    assert q.shape == (6, m.time_axis.n, 3) and np.all(np.isfinite(q))
    wq, wc = member_loop(sb, m, base, members, ip)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)
    assert not np.array_equal(q[0], q[3])   # the members differ


@pytest.mark.parametrize("stack", ["pt_gs_k", "hbv_stack"])
@pytest.mark.parametrize("window, start, steps", [(97, 0, 0), (720, 50, 300), (97, 50, 300)])
def test_windows_and_ranges(sb, stack, window, start, steps):
    m, base, members, ip = case(sb, stack, E=4, seed=1)
    q, c = m.run_ensemble(ip, members, start_step=start, n_steps=steps, window_steps=window)
    wq, wc = member_loop(sb, m, base, members, ip, start, steps)
    assert q.shape == wq.shape == (4, steps or 720, 3)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)


@pytest.mark.parametrize("stack", ["pt_gs_k", "pt_hs_k", "pt_hps_k"])
def test_override_and_filter(sb, stack):
    m, base, members, ip = case(sb, stack, E=3, seed=2)
    cids = m.catchment_ids
    m.set_catchment_parameter(int(cids[1]), sc.overridden(stack))
    m.set_catchment_calculation_filter([int(cids[0]), int(cids[1])])
    q, c = m.run_ensemble(ip, members, window_steps=200)
    assert np.all(q[:, :, 2] == 0.0) and np.all(c[:, :, 2] == 0.0)     # the filtered catchment's sums stay zero, as in run_cells
    wq, wc = member_loop(sb, m, base, members, ip)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)


@pytest.mark.parametrize("point_fx", ["average", "instant"])
def test_sources_on_a_point_axis(sb, point_fx):
    m, base, members, ip = case(sb, "pt_hs_k", E=4, seed=3, nan=False)
    ta = m.time_axis
    for env in members:
        env.temperature = three_hourly(sb, env.temperature, ta, point_fx)
        env.precipitation = three_hourly(sb, env.precipitation, ta, point_fx)
    q, c = m.run_ensemble(ip, members, window_steps=250)
    wq, wc = member_loop(sb, m, base, members, ip)   # the loop sets them through sb2_set_sources_on_axis
    assert np.array_equal(q, wq) and np.array_equal(c, wc)


def test_members_in_passes(sb):
    """10 000 cells x 21 600 steps of pt_hs_k: 8.7 GB a member, so three members take a pass of two and a pass of one, whose spare copy
    repeats its member.  Each pass launches the step kernel once per chunk of the single path and scatters the state once, the forcing once
    per member and ensemble variable (and once more into the spare copies) and once per variable from the model's own sources"""
    n, days, E = 10000, 900, 3
    m, base, members, ip = case(sb, "pt_hs_k", n=n, days=days, E=E, seed=4, nan=False, radiation_axis=False)
    T = m.time_axis.n
    lay = ec.layout("pt_hs_k", n, 3, T, T, T, E)
    assert (lay["passes"], lay["per_pass"]) == (2, 2) and ec.pass_sizes(E, 2) == [2, 1]
    box = {}
    ks = launched(lambda: box.update(r=m.run_ensemble(ip, members, window_steps=T)))
    chunks = sc.run_cells_chunks(T)
    assert sum(k.startswith("hbv_run_kernel") for k, _ in ks) == lay["passes"] * len(chunks)
    want = sum(1 + 2 * ne + (2 if ne < lay["per_pass"] else 0) + 3 for ne in ec.pass_sizes(E, lay["per_pass"]))
    assert sum(k.startswith("ensemble_scatter_kernel") for k, _ in ks) == want
    q, c = box["r"]
    wq, wc = member_loop(sb, m, base, members, ip)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)


def test_the_kept_region_follows_the_model(sb):
    """the member region is kept between calls: a changed parameter set, override, filter, state or time axis is taken up by the next call"""
    from shyft_b200 import synthetic
    m, base, members, ip = case(sb, "hbv_stack", E=4, seed=11, radiation_axis=False)
    q0, _ = m.run_ensemble(ip, members)
    assert np.array_equal(m.run_ensemble(ip, members)[0], q0)
    cids = m.catchment_ids
    m.set_region_parameter(sc.overridden("hbv_stack"))
    m.set_catchment_parameter(int(cids[0]), sc.DEFAULT["hbv_stack"])
    m.set_catchment_calculation_filter([int(cids[0]), int(cids[2])])
    st = synthetic.default_state(2, m.size()); st[:, 12] = 80.0
    m.set_states(st)
    q, c = m.run_ensemble(ip, members, window_steps=300)
    assert not np.array_equal(q, q0)
    wq, wc = member_loop(sb, m, base, members, ip)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)
    # a shorter axis: the sources go with it and are set again
    ta = m.time_axis
    short = sb.TimeAxis(ta.start + 24 * ta.delta_t, ta.delta_t, ta.n - 48)
    cut = lambda src: (src[0], src[1][24:24 + short.n])
    m.initialize_cell_environment(short)
    base2 = sb.RegionEnvironment(**{k: cut(getattr(base, k)) for k in NAMES})
    m._set_sources(base2)
    m.set_states(st)
    members2 = [sb.RegionEnvironment(temperature=cut(e.temperature), precipitation=cut(e.precipitation)) for e in members]
    q, c = m.run_ensemble(ip, members2)
    wq, wc = member_loop(sb, m, base2, members2, ip)
    assert q.shape == (4, short.n, 3) and np.array_equal(q, wq) and np.array_equal(c, wc)


def test_one_step_launch_for_all_members(sb):
    counts = {}
    for E in (1, 6):
        m, base, members, ip = case(sb, "hbv_stack", E=E, seed=5)
        m.run_ensemble(ip, members)   # warm: plans and kriging operators
        ks = launched(lambda: m.run_ensemble(ip, members))
        counts[E] = [k for k, _ in ks if k.startswith(("hbv_run_kernel", "catchment_reduce_kernel"))]
    assert counts[1] == counts[6] == ["hbv_run_kernel<true,true>", "catchment_reduce_kernel"]


def test_member_against_the_oracle(sb, oracle):
    """member 1 equals the loop bit for bit, and the loop's run of member 1 holds the end-to-end census against the oracle's interpolation
    and run (DESIGN.md section 2): every forcing value within 1e-11, every cell-step without a decision flip within 1e-9; the catchments
    none of whose cells diverged are within 1e-9 at every step"""
    from e2e_cases import oracle_forcing
    from e2e_census import Census
    from parity import assert_parity
    from shyft_b200 import synthetic
    m, base, members, ip = case(sb, "pt_hs_k", E=2, seed=6, nan=False, radiation_axis=False, start=SUMMER)
    q, _ = m.run_ensemble(ip, members)
    wq, _ = member_loop(sb, m, base, members[1:], ip)   # leaves member 1's forcing and series in the model
    assert np.array_equal(q[1], wq[0])
    env = sb.RegionEnvironment(**{k: getattr(members[1], k) or getattr(base, k) for k in NAMES})
    gm, f = oracle_forcing(oracle, m.geo, m.time_axis, env, btk_temperature=True)
    st0 = synthetic.default_state(1, m.size())
    want = oracle.pthsk_run_cells(gm, sc.DEFAULT["pt_hs_k"], f, st0, m.time_axis.start * 10**6, m.time_axis.delta_t * 10**6, ncore=8)
    want.pop("state")
    got = {k: m.response(k) for k in sc.responses("pt_hs_k") if k in want}
    cs = Census(want, f, tx=sc.DEFAULT["pt_hs_k"][5])
    cs.add_window(0, got, {k: m.cell_forcing(k) for k in NAMES})
    r = cs.result()
    assert all(v == 0 for v in r["forcing_outside_1e-11"].values()), r["forcing_outside_1e-11"]
    assert r["cell_steps_within"] >= 0.98, r
    diverged = np.zeros(m.size(), dtype=bool)
    for b in cs.bad.values():
        diverged |= b.any(axis=0)
    cix = m.cell_catchment_ix()
    clean = [k for k in range(3) if not diverged[cix == k].any()]
    assert clean, r
    ref = np.stack([want["avg_discharge"][:, cix == k].sum(axis=1) for k in range(3)], axis=1)
    assert_parity(q[1][:, clean], ref[:, clean], "member 1 catchment discharge, catchments without a divergence", rtol=1e-9)


def test_the_model_is_left_as_it_was(sb):
    m, base, members, ip = case(sb, "pt_gs_k", E=3, seed=7)
    cids = m.catchment_ids
    m.set_catchment_parameter(int(cids[2]), sc.overridden("pt_gs_k"))
    m.interpolate(ip, base, best_effort=False)
    m.run_cells()
    before = dict(state=m.get_states(), initial=m.initial_state, region=m.get_region_parameter(), catch=m.get_catchment_parameter(int(cids[2])),
                  q=m.catchment_discharges(), c=m.catchment_charges(), resp=m.response("avg_discharge"),
                  src={k: m.sources_on_model_axis(k) for k in NAMES}, forcing={k: m.cell_forcing(k) for k in NAMES})
    k0 = m.kernel_launches()
    ks = launched(lambda: m.run_ensemble(ip, members, window_steps=300))
    # every kernel the call launched is counted (the profiler window opens with sb2_unit_eval kernels of no model)
    assert m.kernel_launches() - k0 == sum(not k.startswith("unit_eval_kernel") for k, _ in ks)
    after = dict(state=m.get_states(), initial=m.initial_state, region=m.get_region_parameter(), catch=m.get_catchment_parameter(int(cids[2])),
                 q=m.catchment_discharges(), c=m.catchment_charges(), resp=m.response("avg_discharge"),
                 src={k: m.sources_on_model_axis(k) for k in NAMES}, forcing={k: m.cell_forcing(k) for k in NAMES})
    for k, v in before.items():
        if isinstance(v, dict):
            for kk in v:
                assert np.array_equal(v[kk], after[k][kk], equal_nan=True), (k, kk)
        else:
            assert np.array_equal(v, after[k], equal_nan=True), k


def test_errors(sb):
    from shyft_b200 import capi
    import ctypes as C
    m, base, members, ip = case(sb, "pt_hs_k", E=3, seed=8)
    L, h = m._L, m._h
    xyz, v = members[0].temperature
    vals = np.ascontiguousarray(np.stack([members[e].temperature[1] for e in range(3)]))
    assert L.sb2_set_ensemble_sources(h, 0, C.c_int64(3), C.c_int64(9), capi.dptr(np.ascontiguousarray(xyz)), capi.dptr(vals)) == 0
    pv = np.ascontiguousarray(np.stack([members[e].precipitation[1] for e in range(2)]))
    assert L.sb2_set_ensemble_sources(h, 1, C.c_int64(2), C.c_int64(9), capi.dptr(np.ascontiguousarray(xyz)), capi.dptr(pv)) != 0
    msg = L.sb2_last_error(h).decode()
    assert "2 members" in msg and "3" in msg, msg
    with pytest.raises(RuntimeError, match="wind_speed"):
        m.run_ensemble(ip, [sb.RegionEnvironment(wind_speed=base.wind_speed), sb.RegionEnvironment()])
    with pytest.raises(RuntimeError, match="temperature"):
        m.run_ensemble(ip, [sb.RegionEnvironment(temperature=(xyz, v[:-1])), sb.RegionEnvironment(temperature=(xyz, v))])
    with pytest.raises(RuntimeError, match="precipitation"):
        m.run_ensemble(ip, [sb.RegionEnvironment(precipitation=sb.GeoPointSourceVector([])), sb.RegionEnvironment()])
    with pytest.raises(RuntimeError, match="no ensemble sources"):
        m.run_ensemble(ip, [sb.RegionEnvironment()])
    with pytest.raises(RuntimeError, match="start_step must in range"):
        m.run_ensemble(ip, members, start_step=m.time_axis.n)
    with pytest.raises(RuntimeError, match="start_step\\+n_steps must be within"):
        m.run_ensemble(ip, members, start_step=10, n_steps=m.time_axis.n)
    with pytest.raises(RuntimeError, match="window_steps must be positive"):
        m.run_ensemble(ip, members, window_steps=0)
    bad = [sb.RegionEnvironment(temperature=(xyz, np.full_like(v, np.nan) if e == 1 else v)) for e in range(2)]
    with pytest.raises(RuntimeError, match="No valid sources for time period, giving up."):
        m.run_ensemble(ip, bad)
    m.run_ensemble(ip, members[:2])   # the model still runs after the errors
    m.initialize_cell_environment(m.time_axis)   # drops ensemble sources, as it drops sources
    q = np.zeros((1, 720, 3))
    assert L.sb2_run_ensemble(h, C.byref(ip), 0, 0, 4096, capi.dptr(q), None) != 0
    assert "no ensemble sources" in L.sb2_last_error(h).decode()


def test_red_zones_stay_intact():
    env = dict(os.environ, SB2_GUARD="1")
    prog = f"""
import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
import numpy as np
import shyft_b200 as sb
from shyft_b200 import capi
from test_gpu_ensemble import case, member_loop
for stack, window in (("pt_gs_k", 97), ("hbv_stack", 720)):
    m, base, members, ip = case(sb, stack, E=5, seed=9)
    q, c = m.run_ensemble(ip, members, window_steps=window)
    wq, wc = member_loop(sb, m, base, members, ip)
    assert np.array_equal(q, wq) and np.array_equal(c, wc)
v, msg = capi.check_guards()
print('ensemble ok', 'guards', v, msg)
sys.exit(1 if v else 0)
"""
    r = subprocess.run([sys.executable, "-c", prog], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "ensemble ok" in r.stdout and "guards 0" in r.stdout


def test_pybind_module_and_shim_give_the_ctypes_result(sb):
    from shyft_b200 import _build
    _build.build_pybind_module()
    from shyft_b200 import _shyft_b200_cpp as cpp
    m, base, members, ip = case(sb, "hbv_stack", E=3, seed=10, radiation_axis=False)
    q, c = m.run_ensemble(ip, members, start_step=24, n_steps=200, window_steps=64)
    ta = m.time_axis
    b = cpp.HbvModel(m.geo, list(sc.DEFAULT["hbv_stack"]))
    env = {k: getattr(base, k) for k in NAMES}
    assert b.run_interpolation(ta.start * 10**6, ta.delta_t * 10**6, ta.n, env)
    b.set_states(m.get_states())
    dicts = [{k: v for k, v in (("temperature", e.temperature), ("precipitation", e.precipitation))} for e in members]
    bq, bc = b.run_ensemble(dicts, start_step=24, n_steps=200, window_steps=64)
    assert np.array_equal(bq, q.transpose(0, 2, 1)) and np.array_equal(bc, c.transpose(0, 2, 1))
