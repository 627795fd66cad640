"""The exact goal and statistics references (tests/goal_reference.py) against the oracle's restatement of the reference formulas, and
their teeth: on the GPU tests' own case shapes, each plausible slip of a kernel moves the result by at least ten times the bound the
GPU tests allow."""
import math

import numpy as np
import pytest

import goal_reference as G

H = 3600 * 10**6


def catchment_series(T, K=3, seed=0, charge=False):
    """hourly catchment sums of the shape the GPU tests read back: positive discharge with a daily cycle and events, or a charge that
    changes sign within a day"""
    rng = np.random.default_rng(seed)
    t = np.arange(T)[:, None]
    if charge:
        return np.sin(2 * np.pi * t / 24 + rng.uniform(0, 6, K)) * rng.uniform(0.5, 2, K) + rng.normal(0, 0.1, (T, K))
    return 5 + 2 * np.sin(2 * np.pi * t / 24 + rng.uniform(0, 6, K)) + rng.exponential(1.0, (T, K)) * (rng.random((T, K)) < 0.1) * 20


def period_means(q, cix, first, spp, n):
    v = np.zeros(q.shape[0])
    for c in cix:
        v = v + q[:, c]
    return v[first:first + n * spp].reshape(n, spp).mean(axis=1)


def noisy(x, seed, rel=0.2):
    return x * np.random.default_rng(seed).uniform(1 - rel, 1 + rel, x.size)


# ---- agreement with the oracle ------------------------------------------------------------------------------------------------------
def _assert_within(got, want, bound, what):
    r = G.ratio(got, want, bound)
    assert np.all(r <= 1.0), f"{what}: got {got!r}, exact {want!r} +- {bound!r} (ratio {r})"


@pytest.mark.parametrize("seed", range(6))
def test_goal_formulas_agree_with_the_oracle(oracle, seed):
    rng = np.random.default_rng(seed)
    n = [3, 17, 255, 256, 257, 1000][seed]
    o = rng.normal(10, 3, n)
    m = o * rng.uniform(0.7, 1.3, n)
    if seed % 2:
        o[rng.random(n) < 0.2] = np.nan
        m[rng.random(n) < 0.1] = np.inf
    sim = G.obs_prop(m)
    s = np.abs(m) + rng.uniform(0.1, 1, n)
    sim.scale = [None if x is None else G.Fraction(float(y)) for x, y in zip(sim.value, s)]
    for mode, fn in ((0, oracle.nash_sutcliffe), (2, oracle.abs_diff_sum), (3, oracle.rmse)):
        _assert_within(fn(o, m), *G.goal_exact(mode, o, sim), f"mode {mode}")
    for w in ((1, 1, 1), (1, 0.5, 2), (0, 1, 1), (1, 0, 1), (1, 1, 0)):
        _assert_within(oracle.kling_gupta(o, m, *w), *G.kge_exact(o, sim, *w), f"KGE {w}")
    _assert_within(oracle.abs_diff_sum_scaled(o, m, s), *G.abs_diff_scaled_exact(o, sim), "scaled ABS_DIFF")


def test_goal_formulas_at_the_reference_literals(oracle):
    """test/calibration_test.cpp:561-667 as tests/test_oracle_known_answers.py states them"""
    n = 1000
    i = np.arange(n)
    obs = 10.0 + 5 * np.sin(math.pi * 100.0 * i / n)
    sim = np.where(i < n // 2, obs, 0.0)
    P = G.obs_prop
    assert G.nse_exact(obs, P(obs)) == (0.0, 0.0)
    assert G.nse_exact(obs, P(sim))[0] == pytest.approx(4.5, abs=1e-3)
    assert G.nse_exact([1.0, 10.0, np.nan], P([2.0, 2.0, 2.0]))[0] == pytest.approx((1.0 + 64.0) / (4.5**2 + 4.5**2), abs=1e-12)
    assert G.kge_exact(obs, P(obs))[0] == pytest.approx(0.0, abs=1e-15)
    assert G.kge_exact(obs, P(sim))[0] == pytest.approx(1.0272, abs=1e-4)
    assert G.kge_exact([1.0, 10.0, 1.0], P([2.0, 2.0, 7.0]))[0] == pytest.approx(1.5666, abs=1e-4)
    assert G.kge_exact([1.0, 1.0, 1.0], P([2.0, 2.0, 2.0]), 0.0, 1.0, 0.0)[0] == 1.0
    assert G.abs_diff_exact([1.0, 10.0, 1.0], P([2.0, 2.0, 7.0]))[0] == 15.0
    assert G.abs_diff_exact([1.0, np.nan, 1.0], P([2.0, 2.0, 7.0]))[0] == 7.0
    assert G.rmse_exact([1.0, 10.0, 1.0], P([2.0, 2.0, 7.0]))[0] == pytest.approx(1.4505745987941, rel=1e-13)
    assert G.rmse_exact([1.0, np.nan, 1.0], P([2.0, 2.0, 7.0]))[0] == pytest.approx(4.30116263352131, rel=1e-13)
    # the IEEE classes: no finite pair, a constant obs (NSE x / 0), one pair (KGE's 1 / (n - 1) * 0)
    assert np.isnan(G.nse_exact([np.nan, 1.0], P([1.0, np.nan]))[0]) and np.isnan(G.rmse_exact([np.nan], P([1.0]))[0])
    assert G.abs_diff_exact([np.nan], P([1.0]))[0] == 0.0
    assert G.nse_exact([2.0, 2.0], P([1.0, 3.0]))[0] == math.inf
    assert np.isnan(G.kge_exact([2.0], P([1.0]))[0]) and G.kge_exact([2.0], P([1.0]), 0.0, 1.0, 1.0)[0] == pytest.approx(0.5, abs=0)
    assert np.isnan(G.combine_exact([(np.nan, 0.0), (math.inf, 0.0)], [1.0, 2.0])[0])
    assert G.combine_exact([(1.0, 0.0), (np.nan, 0.0), (4.0, 0.0)], [2.0, 5.0, 1.0])[0] == 2.0


def test_aligned_property_agrees_with_the_oracle_projection(oracle):
    q = catchment_series(24 * 40, seed=1)
    q[100:103, 1] = np.nan                                     # NaN steps: the period average is over the finite ones
    for cix, first, spp, n in (([1], 0, 24, 40), ([2, 0], 5, 3, 300), ([0, 1, 2], 7, 1, 900)):
        v = np.zeros(q.shape[0])
        for c in cix:
            v = v + q[:, c]
        want = oracle.average_to_axis(v, H, first, spp, n)
        p = G.property_exact(q, cix, first, spp, n)
        vals = np.array([np.nan if x is None else float(x) for x in p.value])
        assert np.array_equal(np.isnan(vals), np.isnan(want))
        _assert_within(want, vals, p.err, f"average_to_axis {cix} {spp}")
        sc = oracle.max_abs_average_to_axis(v, H, first, spp, n)
        _assert_within(sc, [np.nan if x is None else float(x) for x in p.scale], p.scale_err, "max_abs")


def test_projection_agrees_with_the_oracle_average_accessor(oracle):
    """random axes, and the literals of test_oracle_resampling.py (time_series_test.cpp:480-571)"""
    T0, DT = 946684800 * 10**6, H
    t = np.array([T0, T0 + DT // 2, T0 + 2 * DT], dtype=np.int64)
    v = np.array([1.0, 2.0, 3.0])
    val, _, _ = G.project_exact(t, v, 10**18, [(T0, T0 + 3 * DT), (T0 + 600 * 10**6, T0 + 660 * 10**6), (T0 + 5 * DT, T0 + 60 * DT),
                                               (T0 - 5 * DT, T0 - 4 * DT)])
    assert val[0] == G.Fraction(1 * 1 + 2 * 3 + 3 * 2, 6) and val[1] == 1 and val[2] == 3 and val[3] is None
    tn = np.array([T0, T0 + DT // 2, T0 + DT, T0 + 2 * DT], dtype=np.int64)
    for vv, want in (([np.nan, 2.0, np.nan, 3.0], (0.5 * 2 + 3.0) / 1.5), ([1.0, 2.0, np.nan, 3.0], (1.0 * 0.5 + 0.5 * 2 + 3.0) / 2.0),
                     ([1.0, 2.0, np.nan, np.nan], (1.0 * 0.5 + 0.5 * 2) / 1.0)):
        assert float(G.project_exact(tn, vv, 10**18, [(T0, T0 + 3 * DT)])[0][0]) == pytest.approx(want, rel=1e-15)
    rng = np.random.default_rng(3)
    for case in range(4):
        n = 200
        tt = T0 + np.cumsum(rng.integers(1, 3 * DT, n)).astype(np.int64)
        vals = rng.normal(0, 5, n)
        vals[rng.random(n) < 0.1] = np.nan
        t_end = int(tt[-1]) + DT
        ta0, tadt = int(tt[0]) - DT + int(rng.integers(-10**6, 10**6)), [1, 1200 * 10**6, DT + 1, 7 * 24 * DT][case]
        m = min(300, (t_end + 2 * DT - ta0) // tadt)
        want = oracle.average_accessor(tt, vals[:, None], t_end, False, ta0, tadt, m)[:, 0]
        got, mag, pieces = G.project_exact(tt, vals, t_end, [(ta0 + i * tadt, ta0 + (i + 1) * tadt) for i in range(m)])
        exact = np.array([np.nan if x is None else float(x) for x in got])
        assert np.array_equal(np.isnan(exact), np.isnan(want)), case
        _assert_within(want, exact, G.gamma(pieces + 4) * mag, f"projection case {case}")


def test_statistics_references_agree_with_the_oracle(oracle):
    rng = np.random.default_rng(8)
    n, T = 300, 20
    X = rng.normal(0, 1, (T, n)) * 10.0 ** rng.integers(-5, 6, (T, n))
    area = 10 ** rng.uniform(3, 8, n)
    cids = 1 + (np.arange(n) % 3)
    sel = np.isin(cids, [1, 3])
    s, b = G.stat_sum_exact(X, sel)
    _assert_within(oracle.sum_catchment_feature(X, cids, [1, 3]), s, b, "sum")
    s, b = G.stat_sum_exact(X, sel, area)
    want = oracle.average_catchment_feature(X, area, cids, [1, 3])
    _assert_within(want, s / area[sel].sum(), b / area[sel].sum() + 4 * G.gamma(n) * np.abs(s / area[sel].sum()), "area average")
    mean, mb = G.area_mean_exact(X, area, np.flatnonzero(sel))
    _assert_within(want, mean, mb, "catchment area mean")
    kd = np.abs(rng.normal(0, 1, (T, n))) * area * 1e-7
    pr, pb = G.pot_ratio_exact(kd, area, 1.5)
    _assert_within(oracle.ae_pot_ratio(kd, area, 1.5), pr, pb * 2, "pot_ratio")      # the oracle's exp and the device's: 1 ulp each
    # the IEEE class of a sum with non-finite terms
    Y = np.ones((4, 5))
    Y[0, 1], Y[1, 2], Y[2, 0], Y[2, 4], Y[3, 3] = np.nan, np.inf, np.inf, -np.inf, -np.inf
    s, b = G.stat_sum_exact(Y, np.ones(5, dtype=bool))
    assert np.isnan(s[0]) and s[1] == np.inf and np.isnan(s[2]) and s[3] == -np.inf and np.all(b == 0)
    s, _ = G.stat_sum_exact(Y, np.array([0, 0, 0, 1, 0], dtype=bool))
    assert list(s) == [1.0, 1.0, 1.0, -np.inf]


# ---- teeth: each slip breaks the bound by at least 10x ---------------------------------------------------------------------------
def _gap(slipped, exact_bound):
    v, b = exact_bound
    assert math.isfinite(v) and math.isfinite(slipped), (v, slipped)
    return abs(slipped - v) / b if b > 0 else math.inf


def _teeth(slipped, exact_bound, what):
    g = _gap(slipped, exact_bound)
    assert g >= 10.0, f"{what}: the slip moves the goal by only {g:.2f} bounds"


# the GPU test's aligned shapes (n, steps per period, first step) and catchment lists; 8 784 hourly steps of 3 catchments
SHAPES = [(2, 168, 8784 - 336), (255, 24, 0), (256, 3, 1), (257, 24, 0), (4097, 2, 590)]
CIX = ([1], [0, 2], [2, 0, 1])


def _drop(p, k, dup=False):
    """the property with period k dropped (it pairs with no obs), or period k counted twice (periods k + 1 .. pair with one period early)"""
    ix = list(range(len(p)))
    if dup:
        ix = ix[:k + 1] + ix[k:-1]
    val = [None if (i == k and not dup) else p.value[j] for i, j in enumerate(ix)]
    return G.Prop(val, p.mag[ix], p.err[ix], [p.scale[j] for j in ix], p.scale_err[ix])


@pytest.mark.parametrize("shape", range(len(SHAPES)))
def test_teeth_periods_modes_and_columns(shape):
    n, spp, first = SHAPES[shape]
    q = catchment_series(8784, seed=shape)
    ch = catchment_series(8784, seed=shape, charge=True)
    cix = CIX[shape % 3]
    obs = noisy(period_means(q, cix, first, spp, n), shape)
    cobs = period_means(ch, cix, first, spp, n) + np.random.default_rng(shape).normal(0, 0.3, n)
    p = G.property_exact(q, cix, first, spp, n)
    pc = G.property_exact(ch, cix, first, spp, n)
    wrong_col = [(cix[0] + 1) % 3] + cix[1:]
    pw = G.property_exact(q, wrong_col, first, spp, n)
    pcw = G.property_exact(ch, wrong_col, first, spp, n)
    k = n - 1 if n > 2 else 0
    for mode in (0, 1, 2, 3, 4):
        o, prop, bad = (cobs, pc, pcw) if mode == 4 else (obs, p, pw)
        exact = G.goal_exact(mode, o, prop)
        ev = lambda x: G.goal_exact(mode, o, x)[0]
        if n > 2 or mode not in (0, 1):                           # one pair left: NSE and KGE are not finite
            _teeth(ev(_drop(prop, k)), exact, f"mode {mode} {SHAPES[shape]}: a period dropped")
            _teeth(ev(_drop(prop, (n - 1) // 2, dup=True)), exact, f"mode {mode} {SHAPES[shape]}: a period duplicated")
        _teeth(ev(bad), exact, f"mode {mode} {SHAPES[shape]}: the wrong catchment column")
    # |mean| in place of the max-abs scale
    s_mean = G.Prop(pc.value, pc.mag, pc.err, [abs(x) for x in pc.value], pc.scale_err)
    _teeth(G.abs_diff_scaled_exact(cobs, s_mean)[0], G.abs_diff_scaled_exact(cobs, pc), "|mean| as the scale")
    # n in place of n - 1 in the covariance (the variances keep n - 1)
    if n > 2:
        _teeth(_kge_cov_over_n(obs, p), G.kge_exact(obs, p), f"KGE {SHAPES[shape]}: n in place of n - 1")


def _kge_cov_over_n(obs, p):
    o = np.asarray(obs)
    m = np.array([float(x) for x in p.value])
    c = o.size
    vx, vy = np.var(o, ddof=1), np.var(m, ddof=1)
    r = (np.mean(o * m) - o.mean() * m.mean()) / math.sqrt(vx * vy)
    a, b = m.mean() / o.mean(), math.sqrt(vy / vx)
    assert c > 2
    return math.sqrt((r - 1) ** 2 + (a - 1) ** 2 + (b - 1) ** 2)


def test_teeth_finite_steps_and_finite_pairs():
    """the period average over the finite steps, not steps_per_period; the NSE mean over the finite pairs, not every finite obs"""
    n, spp, first = 255, 24, 0
    q = catchment_series(8784, seed=11)
    q[1000:1010, 0] = np.nan                                     # a gap of the simulated series inside period 41
    p = G.property_exact(q, [0, 2], first, spp, n)
    obs = noisy(period_means(np.nan_to_num(q), [0, 2], first, spp, n), 11)
    slip = G.Prop(list(p.value), p.mag, p.err, p.scale, p.scale_err)
    i = 1000 // 24
    slip.value[i] = p.value[i] * G.Fraction(24 - 10, 24)         # the finite steps' sum over all 24
    for mode in (0, 1, 2, 3):
        _teeth(G.goal_exact(mode, obs, slip)[0], G.goal_exact(mode, obs, p), f"mode {mode}: / steps_per_period")
    # NSE: obs finite where the projected sim is NaN (periods before the model axis)
    sim = G.obs_prop(np.concatenate([[np.nan] * 3, noisy(obs[3:], 12)]))
    o = obs.copy()
    o[:3] = 1000.0
    exact = G.nse_exact(o, sim)
    mean_all = np.mean(o)
    fin = [i for i in range(n) if sim.value[i] is not None]
    slipped = sum((o[i] - float(sim.value[i])) ** 2 for i in fin) / sum((o[i] - mean_all) ** 2 for i in fin)
    _teeth(slipped, exact, "NSE mean over every finite obs")


def test_teeth_area_weights_and_members():
    """an unweighted area mean (cell areas over 1e3 .. 1e8 m2) and a batch member reading its neighbour's series (one ens_stride off)"""
    rng = np.random.default_rng(5)
    T, n = 24 * 30, 48
    area = np.geomspace(1e3, 1e8, n)
    swe = np.abs(rng.normal(50, 20, (T, n))) * np.linspace(0.5, 1.5, n)
    cells = np.arange(1, n, 2)
    mean, b = G.area_mean_exact(swe, area, cells)
    plain = swe[:, cells].mean(axis=1)
    assert np.min(np.abs(plain - mean) / b) >= 10.0
    # members: parameter sets differ by 1 % in their discharge
    q = catchment_series(8784, seed=3)
    n_p, spp = 257, 24
    obs = noisy(period_means(q, [0, 1], 0, spp, n_p), 3)
    p0 = G.property_exact(q, [0, 1], 0, spp, n_p)
    p1 = G.property_exact(q * 1.01, [0, 1], 0, spp, n_p)
    for mode in (0, 1, 2, 3):
        _teeth(G.goal_exact(mode, obs, p1)[0], G.goal_exact(mode, obs, p0), f"mode {mode}: one ens_stride off")
