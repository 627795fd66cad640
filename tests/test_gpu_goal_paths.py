"""The calibration goal kernels (shyft_b200/csrc/sb2_goal.cuh and the projection kernels of sb2_interp.cuh) against the exact references
of tests/goal_reference.py, at the shapes where they can go wrong.

Each case sets targets, calls calculate_goal_function(p), reads back what the goal kernel consumed (the catchment discharge or charge
sums, the snow responses, a river's output flow) and compares the goal with the exact value computed from those bits, within the bound
the reference derives from the kernel's operation.  The worst error / bound ratio per case is printed at the end of the module.

    aligned     n in {1, 2, 52, 255, 256, 257, 4 097} periods of {1, 2, 3, 24, 168} hourly steps, first period at step 0 or later, 1, 2 and
                all 3 catchments (listed out of order); all five modes (NSE, KGE, ABS_DIFF, RMSE, scaled ABS_DIFF of the charge)
    obs         leading / trailing / interleaved NaN, all but one NaN, all NaN, constant obs, a mean of 1e6 with spread 1, negative
                charge obs, KGE with s_r, s_a or s_b = 0
    unaligned   20-minute periods, a half-step shift, boundaries 1 us off a step, periods before / across the end of / after the model
                axis, a point axis of periods from 5 us to two weeks, scaled ABS_DIFF of the charge there (goal_max_kernel)
    snow        SCA and SWE targets on pt_gs_k over cell areas of 1e3 .. 1e8 m2 and a one-cell catchment; a ROUTED_DISCHARGE target
    multi       three targets with unequal scale factors, one of them not finite
    batch       9 parameter sets x 2 targets: bit-equal to single evaluation, three members against the exact reference
"""
import math
import time

import numpy as np
import pytest

import goal_reference as G
from fixtures import HBV_DEFAULT

pytestmark = pytest.mark.gpu
H = 3600
US = 10**6
DAY = 86400
T = 8784                       # one leap year of hourly steps
START = 1420070400             # 2015-01-01
WINTER = 1424476800            # 2015-02-21
CIX = {1: 0, 2: 1, 3: 2}       # catchment id -> column of the catchment sums (order of first appearance)

WORST = {}


def note(case, r):
    WORST[case] = max(WORST.get(case, 0.0), float(r))


@pytest.fixture(scope="module", autouse=True)
def _report():
    t0 = time.perf_counter()
    yield
    print("\nworst goal error per case, in units of its exact bound (<= 1 passes):")
    for case, r in sorted(WORST.items()):
        print(f"  {case:44s} {r:.3e}")
    print(f"module wall time {time.perf_counter() - t0:.1f} s")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


@pytest.fixture(scope="module")
def hbv(sb):
    """64 hbv_stack cells in 3 catchments (22, 22, 20 cells), routed by a chain of 3 rivers, a leap year of hourly steps"""
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(64, T, 4, config_index=41, cells_per_catchment=22, with_routing=True, start=START)
    m = sb.HbvStackModel(geo, HBV_DEFAULT)
    assert m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(synthetic.default_state(2, 64))
    m.set_river_network(synthetic.river_chain(3))
    m.run_cells()
    return m, ta, m.catchment_discharges().copy(), m.catchment_charges().copy()


def period_means(q, cols, first, spp, n):
    v = np.zeros(q.shape[0])
    for c in cols:
        v = v + q[:, c]
    return v[first:first + n * spp].reshape(n, spp).mean(axis=1)


_PROPS = {}


def aligned_prop(series, cols, first, spp, n):
    key = (series.tobytes().__hash__(), tuple(cols), first, spp, n)
    if key not in _PROPS:
        _PROPS[key] = G.property_exact(series, cols, first, spp, n)
    return _PROPS[key]


def evaluate(sb, m, p, targets, props):
    """calculate_goal_function(p) with `targets`; props[k](Q, C) = the exact property of target k from the read-back catchment sums ->
    (goal, exact goal, bound, partials)"""
    opt = sb.Optimizer(m, targets)
    g = opt.calculate_goal_function(p)
    Q, C = m.catchment_discharges(), m.catchment_charges()
    partials = []
    for t, prop in zip(targets, props):
        mode = 4 if (t.calc_mode == 2 and t.catchment_property == 4) else t.calc_mode
        partials.append(G.goal_exact(mode, t.values, prop(Q, C), t.s_r, t.s_a, t.s_b))
    want, bound = G.combine_exact(partials, [t.scale_factor for t in targets])
    return g, want, bound, partials


def check(case, sb, m, p, targets, props):
    g, want, bound, partials = evaluate(sb, m, p, targets, props)
    r = G.ratio(g, want, bound)[0]
    note(case, r)
    assert r <= 1.0, f"{case}: goal {g!r}, exact {want!r} +- {bound:.3e} ({r:.2f} bounds); partials {partials}"
    return g, want, partials


def target(sb, obs, first, spp, cids, mode, charge=False, sf=1.0, **kw):
    return sb.TargetSpecification(obs, START + first * H, spp * H, cids, sf, 2 if mode == 4 else mode,
                                  catchment_property=4 if (charge or mode == 4) else 0, **kw)


# ---- aligned targets -------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1, 0), (1, 168, 5000), (2, 3, 0), (2, 168, T - 336), (52, 168, 48), (255, 24, 0), (256, 24, 17), (257, 24, 0),
          (256, 3, 1), (257, 1, T - 257), (4097, 1, 0), (4097, 2, 590)]
CIDS = ([2], [1, 3], [3, 1, 2])


@pytest.mark.parametrize("shape", SHAPES, ids=[f"n{n}_spp{s}_at{f}" for n, s, f in SHAPES])
def test_aligned_targets_all_modes(sb, hbv, shape):
    m, ta, Q0, C0 = hbv
    n, spp, first = shape
    assert first + n * spp <= T
    cid_sets = CIDS if n in (257, 4097) else (CIDS[SHAPES.index(shape) % 3],)
    rng = np.random.default_rng(n * 7 + spp)
    for cids in cid_sets:
        cols = [CIX[c] for c in cids]
        obs = period_means(Q0, cols, first, spp, n) * rng.uniform(0.8, 1.2, n)
        cobs = period_means(C0, cols, first, spp, n) + rng.normal(0, 0.2, n)
        for mode in range(5):
            o = cobs if mode == 4 else obs
            use_c = mode == 4
            t = target(sb, o, first, spp, cids, mode)
            g, want, _ = check(f"aligned n={n} spp={spp}", sb, m, HBV_DEFAULT, [t],
                               [lambda Q, C: aligned_prop(C if use_c else Q, cols, first, spp, n)])
            if n == 1 and mode in (0, 1):
                assert np.isnan(g)                                 # one period: NSE 0 / 0 or x / 0, KGE 1 / (n - 1) * 0; dropped


# ---- observation patterns ----------------------------------------------------------------------------------------------------------------
def _obs_cases(Q0, C0, cols, first, spp, n):
    rng = np.random.default_rng(5)
    base = period_means(Q0, cols, first, spp, n) * rng.uniform(0.8, 1.2, n)
    lead_trail = base.copy()
    lead_trail[:20] = np.nan
    lead_trail[-15:] = np.nan
    lead_trail[40:200:3] = np.nan
    one = np.full(n, np.nan)
    one[123] = base[123]
    return {"lead, trail, interleaved NaN": lead_trail, "all but one NaN": one, "all NaN": np.full(n, np.nan),
            "constant 5.0": np.full(n, 5.0), "mean 1e6 spread 1": 1e6 + rng.normal(0, 1, n)}


def test_observation_patterns(sb, hbv):
    m, ta, Q0, C0 = hbv
    n, spp, first = 300, 24, 24
    cids = [1, 2]
    cols = [0, 1]
    prop = lambda Q, C: aligned_prop(Q, cols, first, spp, n)
    for name, obs in _obs_cases(Q0, C0, cols, first, spp, n).items():
        for mode in range(4):
            g, want, partials = check(f"obs {name}", sb, m, HBV_DEFAULT, [target(sb, obs, first, spp, cids, mode)], [prop])
            if name == "all NaN":
                assert (g == 0.0) if mode == 2 else np.isnan(g)    # no pair: ABS_DIFF sums nothing; the rest are 0 / 0, dropped
            if name == "constant 5.0" and mode in (0, 1):
                assert np.isnan(g) and not math.isfinite(partials[0][0])   # NSE x / 0; KGE r = x / 0: dropped, the goal is 0 / 0
        if name == "constant 5.0":                                 # KGE without r: b = us / 0 is set to 1
            g, want, _ = check("obs constant, KGE s_r = 0", sb, m, HBV_DEFAULT, [target(sb, obs, first, spp, cids, 1, s_r=0.0)], [prop])
            assert math.isfinite(g)
    # an all-NaN target next to a finite one is dropped from the weighted mean
    base = _obs_cases(Q0, C0, cols, first, spp, n)["lead, trail, interleaved NaN"]
    g, want, partials = check("obs all NaN dropped", sb, m, HBV_DEFAULT,
                              [target(sb, np.full(n, np.nan), first, spp, cids, 0, sf=2.0), target(sb, base, first, spp, cids, 3, sf=0.5)],
                              [prop, prop])
    assert g == pytest.approx(partials[1][0], rel=1e-15)
    # KGE with each weight zero
    for w in ((0.0, 1.0, 1.0), (1.0, 0.0, 1.0), (1.0, 1.0, 0.0), (2.0, 0.5, 0.0)):
        check("obs KGE weights", sb, m, HBV_DEFAULT, [target(sb, base, first, spp, cids, 1, s_r=w[0], s_a=w[1], s_b=w[2])], [prop])
    # negative charge obs: the scaled ABS_DIFF over max-abs scales
    cobs = -np.abs(period_means(C0, cols, first, spp, n)) - 0.5
    check("obs negative charge, scaled", sb, m, HBV_DEFAULT, [target(sb, cobs, first, spp, cids, 4)],
          [lambda Q, C: aligned_prop(C, cols, first, spp, n)])


# ---- targets not aligned with the model axis -------------------------------------------------------------------------------------------
def _names(kernels):
    return [k for k, _ in kernels]


def test_unaligned_targets_take_the_projection_kernels(sb, hbv):
    from test_gpu_step_paths import launched
    m, ta, Q0, C0 = hbv
    t_us = (START + H * np.arange(T, dtype=np.int64)) * US
    t_end = (START + H * T) * US
    rng = np.random.default_rng(9)
    cids, cols = [3, 1], [2, 0]

    def fixed(t0_s, dt_s, n):
        return [((t0_s + i * dt_s) * US, (t0_s + (i + 1) * dt_s) * US) for i in range(n)]

    def obs_for(periods, charge=False):
        p = G.projected_prop(t_us, C0 if charge else Q0, cols, t_end, periods)
        v = np.array([np.nan if x is None else float(x) for x in p.value])
        return (np.where(np.isfinite(v), v, 1.0) + rng.normal(0, 0.3, v.size)) if charge else np.where(np.isfinite(v), v, 1.0) * rng.uniform(0.8, 1.2, v.size)

    cases = [("20-minute periods", START + 5 * H, 1200, 600), ("half-step shift", START + 1800, 3 * H, 400),
             ("before, across and after the axis", START - 3 * DAY - 900, DAY, 372)]
    for name, t0_s, dt_s, n in cases:
        periods = fixed(t0_s, dt_s, n)
        obs = obs_for(periods)
        for mode in range(4):
            t = sb.TargetSpecification(obs, t0_s, dt_s, cids, 1.0, mode)
            prop = lambda Q, C, periods=periods: G.projected_prop(t_us, Q, cols, t_end, periods)
            ks = launched(lambda: check(f"unaligned {name}", sb, m, HBV_DEFAULT, [t], [prop]))
            assert "goal_property_kernel" in _names(ks) and "average_accessor_kernel" in _names(ks) and "goal_kernel" in _names(ks), ks
    # point axes: boundaries 1 us off a step, and periods from 5 us to two weeks
    base = (START + 100 * H) * US
    off = [base + k * H * US + (1 if k % 2 else -1) for k in range(200)]
    gaps = np.array([5, 1, 10**6, H * US, H * US + 1, 1800 * US, DAY * US, 7 * DAY * US, 14 * DAY * US, 37], dtype=np.int64)
    free = base + np.concatenate([[0], np.cumsum(np.tile(gaps, 6))])
    free = free[free < t_end + 3 * DAY * US]
    for name, pts in (("points 1 us off a step", np.array(off, dtype=np.int64)), ("points 5 us .. two weeks", free)):
        periods = list(zip(pts[:-1], pts[1:]))
        obs = obs_for(periods)
        for mode in (0, 2, 3):
            t = sb.TargetSpecification(obs, 0, 0, cids, 1.0, mode, time_points=pts / US)
            assert np.array_equal(t.time_points_us, pts)
            prop = lambda Q, C, periods=periods: G.projected_prop(t_us, Q, cols, t_end, periods)
            ks = launched(lambda: check(f"unaligned {name}", sb, m, HBV_DEFAULT, [t], [prop]))
            assert "average_accessor_periods_kernel" in _names(ks), ks
        # scaled ABS_DIFF of the charge on such an axis: max of the projected max(0, v) and max(0, -v)
        cobs = obs_for(periods, charge=True)
        t = sb.TargetSpecification(cobs, 0, 0, cids, 1.0, 2, catchment_property=4, time_points=pts / US)
        prop = lambda Q, C, periods=periods: G.projected_prop(t_us, C, cols, t_end, periods, scaled=True)
        ks = launched(lambda: check(f"unaligned {name}, scaled charge", sb, m, HBV_DEFAULT, [t], [prop]))
        assert "goal_max_kernel" in _names(ks) and _names(ks).count("average_accessor_periods_kernel") == 3, ks


# ---- several targets, a routed target, a batch ------------------------------------------------------------------------------------------
def test_weighted_targets_and_a_routed_target(sb, hbv):
    from test_gpu_step_paths import launched
    m, ta, Q0, C0 = hbv
    rng = np.random.default_rng(13)
    o1 = period_means(Q0, [0], 0, 24, 366) * rng.uniform(0.8, 1.2, 366)
    o2 = period_means(Q0, [1, 2], 6, 6, 1000) * rng.uniform(0.8, 1.2, 1000)
    targets = [target(sb, o1, 0, 24, [1], 0, sf=2.0), target(sb, o2, 6, 6, [2, 3], 3, sf=0.5),
               target(sb, np.full(100, 5.0), 0, 24, [3], 0, sf=1.25)]
    props = [lambda Q, C: aligned_prop(Q, [0], 0, 24, 366), lambda Q, C: aligned_prop(Q, [1, 2], 6, 6, 1000),
             lambda Q, C: aligned_prop(Q, [2], 0, 24, 100)]
    ks = launched(lambda: check("three targets, one not finite", sb, m, HBV_DEFAULT, targets, props))
    assert [g for k, g in ks if k == "goal_kernel"][0][:2] == [3, 1], ks
    # ROUTED_DISCHARGE: the per-target series path (n_col 1) over the river's output flow
    rid = 3
    obs = period_means(Q0, [0, 1, 2], 0, 24, 300) * rng.uniform(0.8, 1.2, 300)
    for mode in range(4):
        t = sb.TargetSpecification(obs, START, DAY, [], 1.0, mode, catchment_property=3, river_id=rid)
        g = sb.Optimizer(m, [t]).calculate_goal_function(HBV_DEFAULT)
        want, bound = G.goal_exact(mode, obs, G.property_exact(m.river_output_flow_m3s(rid)[:, None], [0], 0, 24, 300))
        r = G.ratio(g, want, bound)[0]
        note("routed discharge", r)
        assert r <= 1.0, (mode, g, want, bound)


def test_batch_members_equal_single_and_the_exact_goal(sb, hbv):
    m, ta, Q0, C0 = hbv
    rng = np.random.default_rng(21)
    o1 = period_means(Q0, [0, 1], 0, 24, 366) * rng.uniform(0.8, 1.2, 366)
    o2 = period_means(Q0, [2], 3, 6, 1400) * rng.uniform(0.8, 1.2, 1400)
    targets = [target(sb, o1, 0, 24, [1, 2], 0, sf=1.0), target(sb, o2, 3, 6, [3], 1, sf=3.0, s_a=0.5, s_b=2.0)]
    P = np.tile(HBV_DEFAULT, (9, 1))
    P[:, 0] = rng.uniform(150.0, 450.0, 9)     # soil.fc
    P[:, 1] = rng.uniform(1.0, 4.0, 9)         # soil.beta
    P[:, 4] = rng.uniform(0.2, 0.7, 9)         # tank.kuz2
    P[:, 13] = rng.uniform(0.8, 1.4, 9)        # p_corr
    opt = sb.Optimizer(m, targets)
    batch = opt.calculate_goal_function_batch(P)
    single = np.array([opt.calculate_goal_function(p) for p in P])
    assert np.array_equal(batch, single)
    props = [lambda Q, C: aligned_prop(Q, [0, 1], 0, 24, 366), lambda Q, C: aligned_prop(Q, [2], 3, 6, 1400)]
    for i in (0, 4, 8):
        g, want, _ = check("batch members via single", sb, m, P[i], targets, props)
        assert g == batch[i]


# ---- snow targets on pt_gs_k ---------------------------------------------------------------------------------------------------------
def test_snow_targets_over_uneven_areas(sb):
    from shyft_b200 import synthetic

    from test_gpu_step_paths import launched
    n, TT = 48, 24 * 60
    geo, ta, env = synthetic.make_region(n, TT, 4, config_index=43, cells_per_catchment=n, start=WINTER)
    geo["area"] = np.geomspace(1e3, 1e8, n)[np.random.default_rng(2).permutation(n)]
    geo["catchment_id"] = np.where(np.arange(n) == 5, 1, 2 + np.arange(n) % 2)      # catchment 1: one cell
    m = sb.PTGSKModel(geo)
    assert m.run_interpolation(sb.InterpolationParameter(), ta, env)
    st = synthetic.default_state(0, n)
    st[:, 5] = -1.0
    st[:, 4] = np.linspace(5.0, 80.0, n)
    m.set_states(st)
    p = m.get_region_parameter()
    area, cid = np.asarray(geo["area"]), np.asarray(geo["catchment_id"])
    rng = np.random.default_rng(4)
    for prop_id, resp in ((1, "snow_sca"), (2, "snow_swe")):
        m.run_cells()
        v0 = m.response(resp)
        for cids, mode, spp, first, nper in (([1], 3, 24, 0, 60), ([2, 3], 0, 6, 2, 230), ([3], 1, 24, 24, 59), ([2], 2, 1, 0, TT)):
            if mode == 1 and resp == "snow_sca":
                continue                                         # a fully snow-covered catchment has no SCA variance for KGE's r
            cells = np.flatnonzero(np.isin(cid, cids))
            w = area[cells]
            mean0 = (v0[:, cells] * w).sum(axis=1) / w.sum()
            obs = mean0[first:first + nper * spp].reshape(nper, spp).mean(axis=1) * rng.uniform(0.9, 1.1, nper) + 0.01
            t = sb.TargetSpecification(obs, ta.start + first * H, spp * H, cids, 1.0, mode, catchment_property=prop_id)
            opt = sb.Optimizer(m, [t])
            ks = launched(lambda: opt.calculate_goal_function(p))
            g = opt.goal_fn_trace[-1]
            assert "catchment_area_mean_kernel" in _names(ks), ks
            vals, err, mag = G.area_mean_series(m.response(resp), area, cells)
            want, bound = G.goal_exact(mode, obs, G.series_prop(vals, err, mag, first, spp, nper))
            r = G.ratio(g, want, bound)[0]
            note(f"snow {resp} ({'one cell' if cids == [1] else 'cells of 1e3..1e8 m2'})", r)
            assert r <= 1.0, (resp, cids, mode, g, want, bound)
