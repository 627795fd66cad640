"""Exact references of the calibration goal kernels (shyft_b200/csrc/sb2_goal.cuh, the projection of sb2_interp.cuh) and of the
statistics readers (sb2_stats.cuh).

Every function takes the float64 inputs the device kernel read (catchment sums, projected series, per-cell rows) and evaluates the
operation exactly: sums and means of doubles in fractions.Fraction, square roots and exp in mpmath at 40 digits.  Each result comes
with an absolute error bound derived from the operation, never a relative tolerance (a twin target has goal 0):

- a sum of m float64 terms, in any order and tree, is within gamma(m - 1) * sum|terms| of the exact sum (Higham, ASNA 4.2); the
  kernels sum in a known depth: per-thread strides + 8 tree levels (goal_kernel), + 5 shuffle levels + 8 warp parts
  (stat_reduce_rows_kernel), the inner period loop and the catchment columns (the aligned property);
- each further multiply, divide or sqrt adds one unit round-off u = 2^-53 relative to its result;
- errors of the inputs of a formula are carried to first order through its derivative, with absolute values, and that is where the
  cancellations of the formulas show: KGE's sxx - sx^2 / n, RMSE's division by the obs mean, NSE's division by the obs spread.

The semantics are those of the reference (oracle/sho_region.hpp goal::*, core/time_series.h:2316-2448):
only pairs with both values finite count; the NSE mean is taken over those pairs; KGE uses n - 1 denominators (dlib's
running_scalar_covariance) and sets a or b to 1 when it is not finite; scaled ABS_DIFF skips |scale| <= 1e-20.
A non-finite exact result is returned as the IEEE value (NaN or +-inf) that the same operation gives on exact values, with bound 0.
"""
import math
from fractions import Fraction

import numpy as np
from mpmath import mp, mpf

from routing_reference import U, exact_sum
from step_cases import gamma

DPS = 40
NAN = float("nan")
TREE = 8                                 # goal_kernel: log2(256) levels of the shared-memory tree
STAT_TREE = 5 + 8                        # stat_reduce_rows_kernel: 5 shuffle levels and the sum of 8 warp parts
K_MMH_M3S = 1 / (3600.0 * 1000.0)        # m3s_to_mmh's constant, as the device holds it


def _div(a, b):
    """a / b of exact values with IEEE's answer for a zero divisor"""
    if b == 0:
        return NAN if (a == 0 or a != a) else math.copysign(math.inf, float(a))
    return a / b


def _f(x):
    """an exact value (Fraction or mpf) rounded to float64; non-finite floats pass through"""
    if isinstance(x, float):
        return x
    return float(x)


def _sqrt(x):
    """sqrt of an exact non-negative value at DPS digits; NaN for a negative one (IEEE)"""
    if x != x or x < 0:
        return NAN
    if x == math.inf:
        return math.inf
    with mp.workdps(DPS):
        return mp.sqrt(mpf(x.numerator) / x.denominator) if isinstance(x, Fraction) else mp.sqrt(mpf(x))


def _mp(x):
    """an exact value as an mpf at the working precision"""
    return mpf(x.numerator) / x.denominator if isinstance(x, Fraction) else mpf(x)


# ---- the simulated property on the target axis ---------------------------------------------------------------------------------------
class Prop:
    """a target's simulated property per target period: value (Fraction, or None where no finite step falls in the period), mag (the
    period mean of the summed |terms|), err (its error bound as the device computes it) and the same three for the max-abs scale"""

    def __init__(self, value, mag, err, scale, scale_err):
        self.value, self.mag, self.err, self.scale, self.scale_err = value, np.asarray(mag), np.asarray(err), scale, np.asarray(scale_err)

    def __len__(self):
        return len(self.value)


def property_exact(series, cix, first_step, steps_per_period, n, dt=3600.0):
    """goal_kernel's aligned property: period i averages steps first_step + i * spp .. + spp - 1 (those inside the series) of the sum of
    the cix columns, over the steps whose float64 sum (in cix order, as the kernel adds) is finite.  The step length dt cancels in the
    exact time-weighted average; it enters the rounding only.  Also max(mean(max(0, v)), mean(max(0, -v))) for the scaled ABS_DIFF."""
    s = np.asarray(series, dtype=np.float64)
    s = s.reshape(s.shape[0], -1)
    T = s.shape[0]
    cix = [int(c) for c in cix]
    fsum_f = np.zeros(T)                                             # the kernel's v: 0.0 + col0 + col1 + ... in cix order
    for c in cix:
        fsum_f = fsum_f + s[:, c]
    depth = len(cix) + steps_per_period + 1                          # columns, v * dt, the period loop, / tsum
    val, mag, err, sc, sc_err = [], [], [], [], []
    for i in range(n):
        a = first_step + i * steps_per_period
        tot, pos, neg, m, k = Fraction(0), Fraction(0), Fraction(0), 0.0, 0
        for t in range(a, min(a + steps_per_period, T)):
            if not math.isfinite(fsum_f[t]):
                continue
            v = sum((Fraction(float(s[t, c])) for c in cix), Fraction(0))
            tot += v
            pos += max(v, 0)
            neg += max(-v, 0)
            m += math.fsum(abs(s[t, c]) for c in cix)
            k += 1
        if k == 0:
            val.append(None)
            sc.append(None)
            mag.append(0.0)
            err.append(0.0)
            sc_err.append(0.0)
            continue
        val.append(tot / k)
        sc.append(max(pos / k, neg / k))
        mag.append(m / k)
        err.append(gamma(depth) * m / k * (1 + 4 * U))
        sc_err.append(gamma(depth + 1) * m / k * (1 + 4 * U))
    return Prop(val, mag, err, sc, sc_err)


def project_exact(t_us, values, t_end_us, periods):
    """average_accessor with linear = 0 (the goal path's projection) over periods [(start_us, end_us)]: point k holds values[k] from t_us[k]
    to t_us[k + 1], the last point up to the period end (flat extension); pieces before the first point, with non-finite values, or in a
    period starting at or after t_end_us do not count.  Returns (value: list of Fraction / None, magnitude, pieces summed) per period."""
    t = [int(x) for x in np.asarray(t_us, dtype=np.int64)]
    v = np.asarray(values, dtype=np.float64)
    out, mags, depth = [], [], []
    for p0, p1 in periods:
        p0, p1 = int(p0), int(p1)
        if not t or p0 >= t_end_us:
            out.append(None), mags.append(0.0), depth.append(0)
            continue
        lo = max(0, int(np.searchsorted(t, p0, side="right")) - 1)
        area, tsum, m, pieces = Fraction(0), 0, 0.0, 0
        for k in range(lo, len(t)):
            if t[k] >= p1:
                break
            a, b = max(t[k], p0), (min(t[k + 1], p1) if k + 1 < len(t) else p1)
            if b <= a or not math.isfinite(v[k]):
                continue
            area += (b - a) * Fraction(float(v[k]))
            tsum += b - a
            m += (b - a) * abs(float(v[k]))
            pieces += 1
        out.append(area / tsum if tsum > 0 else None)
        mags.append(m / tsum if tsum > 0 else 0.0)
        depth.append(pieces)
    return out, np.array(mags), np.array(depth)


def projected_prop(t_us, series, cix, t_end_us, periods, scaled=False):
    """the property of a target whose axis is not aligned with the model axis: goal_property_kernel's column sum (float64, in cix order:
    exactly what the device forms), projected; the device then takes the projected values as they are (steps_per_period 1, dt 1)"""
    s = np.asarray(series, dtype=np.float64).reshape(len(t_us), -1)
    v = np.zeros(s.shape[0])
    for c in cix:
        v = v + s[:, int(c)]
    val, mag, pieces = project_exact(t_us, v, t_end_us, periods)
    err = gamma(pieces + 4) * mag * (1 + 4 * U) + gamma(max(len(cix) - 1, 0)) * mag   # pieces + seconds, product, / tsum; the column sum
    sc, sc_err = [None] * len(val), np.zeros(len(val))
    if scaled:
        fin = np.isfinite(v)
        pv, pm, pp = project_exact(t_us, np.where(fin, np.maximum(0.0, v), v), t_end_us, periods)
        nv, nm, npc = project_exact(t_us, np.where(fin, np.maximum(0.0, -v), v), t_end_us, periods)
        sc = [None if a is None or b is None else max(a, b) for a, b in zip(pv, nv)]
        sc_err = gamma(np.maximum(pp, npc) + 4) * np.maximum(pm, nm) * (1 + 4 * U) + gamma(max(len(cix) - 1, 0)) * mag
    return Prop(val, mag, err, sc, sc_err)


def obs_prop(values):
    """a float64 series taken as a property without error (a test's own observed values, or a device series read back as such)"""
    v = np.asarray(values, dtype=np.float64)
    val = [Fraction(float(x)) if math.isfinite(x) else None for x in v]
    return Prop(val, np.abs(np.where(np.isfinite(v), v, 0.0)), np.zeros(v.size), [None] * v.size, np.zeros(v.size))


# ---- goal functions ------------------------------------------------------------------------------------------------------------------------
def _pairs(obs, sim):
    o = np.asarray(obs, dtype=np.float64)
    assert o.size == len(sim), (o.size, len(sim))
    idx = [i for i in range(o.size) if math.isfinite(o[i]) and sim.value[i] is not None]
    return o, idx


def _depth(n, extra=0):
    """per-thread stride count + the tree + extra operations of the term"""
    return -(-n // 256) + TREE + extra


def abs_diff_exact(obs, sim):
    """sum |o - m| over the finite pairs -> (value, bound)"""
    o, idx = _pairs(obs, sim)
    g = gamma(_depth(len(o), 2))
    val, mag, err = Fraction(0), 0.0, 0.0
    for i in idx:
        d = Fraction(float(o[i])) - sim.value[i]
        val += abs(d)
        mag += abs(float(d)) + sim.err[i]
        err += sim.err[i]
    return _f(val), (err + g * mag) * (1 + 4 * U)


def abs_diff_scaled_exact(obs, sim):
    """sum |o - m| / s over the finite pairs with a finite scale |s| > 1e-20 (abs_diff_sum_goal_function_scaled)"""
    o, idx = _pairs(obs, sim)
    g = gamma(_depth(len(o), 3))
    val, mag, err = Fraction(0), 0.0, 0.0
    for i in idx:
        s = sim.scale[i]
        if s is None or not abs(s) > Fraction(1e-20):
            continue
        d = abs(Fraction(float(o[i])) - sim.value[i])
        q = d / s
        val += q
        fs, fd = float(s), float(d)
        rel_s = sim.scale_err[i] / fs
        assert rel_s < 0.01, "scale too close to its own error for a first-order bound"
        err += (sim.err[i] + fd * rel_s) / fs * (1 + 2 * rel_s)
        mag += float(q) + sim.err[i] / fs
    return _f(val), (err + g * mag) * (1 + 4 * U)


def _sums(obs, sim, idx, depth):
    """the kernel's pass-1 sums with their error bounds: sx, sy, sxx, syy, sxy, sd2 (= sum (o - m)^2) and n"""
    g = gamma(depth)
    S = dict(sx=Fraction(0), sy=Fraction(0), sxx=Fraction(0), syy=Fraction(0), sxy=Fraction(0), sd2=Fraction(0))
    E = dict.fromkeys(S, 0.0)
    M = dict.fromkeys(S, 0.0)
    for i in idx:
        o, m, e = Fraction(float(obs[i])), sim.value[i], sim.err[i]
        fo, fm = abs(float(o)), abs(float(m))
        d = o - m
        fd = abs(float(d))
        S["sx"] += o; M["sx"] += fo
        S["sy"] += m; M["sy"] += fm; E["sy"] += e
        S["sxx"] += o * o; M["sxx"] += fo * fo
        S["syy"] += m * m; M["syy"] += fm * fm; E["syy"] += 2 * fm * e + e * e
        S["sxy"] += o * m; M["sxy"] += fo * fm; E["sxy"] += fo * e
        S["sd2"] += d * d; M["sd2"] += fd * fd; E["sd2"] += 2 * fd * e + e * e
    for k in S:
        E[k] = (E[k] + g * (M[k] + E[k])) * (1 + 4 * U)
    return S, E, len(idx)


def rmse_exact(obs, sim):
    """sqrt(sum (o - m)^2 / n) / mean(o) over the finite pairs; NaN without one"""
    o, idx = _pairs(obs, sim)
    if not idx:
        return NAN, 0.0
    S, E, c = _sums(o, sim, idx, _depth(len(o), 3))
    mean_o = S["sx"] / c
    if mean_o == 0:
        return _f(_div(_sqrt(S["sd2"] / c), mean_o)), 0.0
    with mp.workdps(DPS):
        r = _sqrt(S["sd2"] / c) / _mp(mean_o)
        mo = abs(float(mean_o))
        e_mo = (E["sx"] / c) * (1 + 2 * U)
        assert e_mo < 0.01 * mo, "obs mean too close to its own error for a first-order bound"
        hi = mp.sqrt(_mp(S["sd2"]) / c + mpf(E["sd2"]) / c) - mp.sqrt(_mp(S["sd2"]) / c)   # the sqrt of an error: no first order at 0
        bound = float(hi) / (mo - e_mo) + abs(float(r)) * (e_mo / (mo - e_mo) + 5 * U)
        return float(r), bound * (1 + 4 * U)


def nse_exact(obs, sim):
    """sum (o - m)^2 / sum (o - mean(o))^2, the mean and both sums over the finite pairs"""
    o, idx = _pairs(obs, sim)
    if not idx:
        return NAN, 0.0
    depth = _depth(len(o), 3)
    S, E, c = _sums(o, sim, idx, depth)
    mean_o = S["sx"] / c
    so2, m2 = Fraction(0), 0.0
    for i in idx:
        d = Fraction(float(o[i])) - mean_o
        so2 += d * d
        m2 += abs(float(d))
    d_mean = (E["sx"] / c + 2 * U * abs(float(mean_o))) * (1 + 4 * U)    # the device's mean: sum, then / n
    e_so2 = (2 * m2 * d_mean + c * d_mean * d_mean + gamma(depth) * (float(so2) + 2 * m2 * d_mean)) * (1 + 4 * U)
    if so2 == 0:
        return _f(_div(S["sd2"], so2)), 0.0
    v = S["sd2"] / so2
    fso2 = float(so2)
    assert e_so2 < 0.01 * fso2, "obs spread too close to its own error for a first-order bound"
    bound = (E["sd2"] + abs(float(v)) * e_so2) / (fso2 - e_so2) + 2 * U * abs(float(v))
    return float(v), bound * (1 + 4 * U)


def kge_exact(obs, sim, s_r=1.0, s_a=1.0, s_b=1.0):
    """sqrt((s_r (r - 1))^2 + (s_a (a - 1))^2 + (s_b (b - 1))^2), r / a / b from dlib's n - 1 (co)variances over the finite pairs; a or b
    = 1 where it is not finite; a term with a zero weight is left out"""
    o, idx = _pairs(obs, sim)
    depth = _depth(len(o), 2)
    S, E, c = _sums(o, sim, idx, depth)
    with mp.workdps(DPS):
        def n_(xx, x, y, exx, ex, ey):
            """xx - x y / n exactly, and its error: the sums' errors, then the product, the division and the subtraction"""
            if c == 0:
                return NAN, 0.0
            v = xx - x * y / c
            fx, fy = abs(float(x)), abs(float(y))
            e = exx + (fx * ey + fy * ex + ex * ey) / c + 3 * U * (abs(float(xx)) + fx * fy / c)
            return v, e * (1 + 4 * U)
        nx, enx = n_(S["sxx"], S["sx"], S["sx"], E["sxx"], E["sx"], E["sx"])
        ny, eny = n_(S["syy"], S["sy"], S["sy"], E["syy"], E["sy"], E["sy"])
        nxy, enxy = n_(S["sxy"], S["sx"], S["sy"], E["sxy"], E["sx"], E["sy"])
        # 1 / (n - 1) * N: n = 1 gives inf * 0 = NaN (N is exactly 0 then), n = 0 NaN
        var_x, var_y = (nx / (c - 1), ny / (c - 1)) if c >= 2 else (NAN, NAN)
        fin = lambda x: not (isinstance(x, float) and not math.isfinite(x))
        terms, errs = [], []
        # r = cov / sqrt(var_x var_y)
        if s_r != 0.0:
            if not (fin(var_x) and fin(var_y)) or var_x == 0 or var_y == 0:
                return NAN, 0.0                                      # 0 / 0, x / 0 or a NaN variance: the goal is not finite
            r = _mp(nxy) / mp.sqrt(_mp(nx) * _mp(ny))
            rel = 0.5 * enx / float(nx) + 0.5 * eny / float(ny)
            assert rel < 0.01, "variances too close to their own errors for a first-order bound"
            dr = enxy / math.sqrt(float(nx) * float(ny)) + abs(float(r)) * (rel * (1 + 2 * rel) + 8 * U)
            terms.append(s_r * (r - 1))
            errs.append(abs(s_r) * (dr + U * (abs(float(r)) + 1)))
        if s_a != 0.0:
            if c == 0 or S["sx"] == 0:
                a, da = mpf(1), 0.0
            else:
                a = _mp(S["sy"]) / _mp(S["sx"])
                fsx = abs(float(S["sx"]))
                assert E["sx"] < 0.01 * fsx
                da = (E["sy"] + abs(float(a)) * E["sx"]) / (fsx - E["sx"]) + 3 * U * abs(float(a))
            terms.append(s_a * (a - 1))
            errs.append(abs(s_a) * (da + U * (abs(float(a)) + 1)))
        if s_b != 0.0:
            if not (fin(var_x) and fin(var_y)) or var_x == 0:
                b, db = mpf(1), 0.0                                  # us / uo not finite: b = 1
            else:
                b = mp.sqrt(_mp(var_y) / _mp(var_x))
                if nx != 0 and ny != 0:
                    rel = 0.5 * enx / float(nx) + 0.5 * eny / float(ny)
                    assert rel < 0.01, "variances too close to their own errors for a first-order bound"
                    db = abs(float(b)) * (rel * (1 + 2 * rel) + 6 * U)
                else:                                                # var_y exactly 0: b = 0 up to sqrt(error)
                    assert ny == 0 and eny == 0.0, "a sim variance of 0 is only exact when its sums are"
                    db = 0.0
            terms.append(s_b * (b - 1))
            errs.append(abs(s_b) * (db + U * (abs(float(b)) + 1)))
        if not terms:
            return 0.0, 0.0
        val = mp.sqrt(mp.fsum(t * t for t in terms))
        # | |v_hat| - |v| | <= |v_hat - v| (the norm's triangle inequality), then the squares, their sum and the sqrt
        bound = math.sqrt(math.fsum(e * e for e in errs)) + 3 * U * float(val)
        return float(val), bound * (1 + 4 * U)


GOALS = {0: nse_exact, 2: abs_diff_exact, 3: rmse_exact}


def goal_exact(mode, obs, sim, s_r=1.0, s_a=1.0, s_b=1.0):
    """the partial goal value of one target by goal_kernel's calc_mode (4 = ABS_DIFF of a CELL_CHARGE target: the scaled form)"""
    if mode == 1:
        return kge_exact(obs, sim, s_r, s_a, s_b)
    if mode == 4:
        return abs_diff_scaled_exact(obs, sim)
    return GOALS[mode](obs, sim)


def combine_exact(partials, scale_factors):
    """the scale_factor-weighted mean over the targets with a finite partial value: partials = [(value, bound)] -> (goal, bound);
    NaN (0 / 0) when none is finite"""
    num, den, err, mag = Fraction(0), Fraction(0), 0.0, 0.0
    for (v, b), w in zip(partials, scale_factors):
        if math.isfinite(v):
            num += Fraction(w) * Fraction(v)
            den += Fraction(w)
            err += abs(w) * b
            mag += abs(w * v)
    if den == 0:
        return NAN, 0.0
    k = 2 * len(partials) + 2
    return float(num / den), (err / float(den) + gamma(k) * (mag + err) / float(den)) * (1 + 4 * U)


# ---- catchment means and the statistics readers ---------------------------------------------------------------------------------------
def area_mean_exact(v, area, cells):
    """catchment_area_mean_kernel: sum v[t][c] area[c] / sum area[c] over the given cells, per row: (value [T], bound [T]); the kernel adds
    cell after cell and multiplies by 1 / sum area"""
    v = np.asarray(v, dtype=np.float64)
    a = np.asarray(area, dtype=np.float64)[list(cells)]
    sa = math.fsum(a)
    out, bound = np.zeros(v.shape[0]), np.zeros(v.shape[0])
    for t in range(v.shape[0]):
        x = v[t, list(cells)]
        if not np.all(np.isfinite(x)):
            out[t] = float(np.sum(x * a))                            # the IEEE class of the float sum
            continue
        num = sum((Fraction(float(p)) * Fraction(float(q)) for p, q in zip(x, a)), Fraction(0))
        out[t] = float(num / sum((Fraction(float(q)) for q in a), Fraction(0)))
        bound[t] = gamma(len(cells) + 3) * math.fsum(np.abs(x) * a) / sa * (1 + 4 * U)
    return out, bound


def area_mean_series(v, area, cells):
    """catchment_area_mean_kernel's per-step series as exact values: (list of Fraction, error bound [T], magnitude [T]); the error of the
    kernel's cell-after-cell sums and its * (1 / sum area)"""
    v = np.asarray(v, dtype=np.float64)[:, list(cells)]
    a = np.asarray(area, dtype=np.float64)[list(cells)]
    fa = [Fraction(float(x)) for x in a]
    den = sum(fa, Fraction(0))
    vals = [sum((Fraction(float(x)) * w for x, w in zip(row, fa)), Fraction(0)) / den for row in v]
    mag = (np.abs(v) * a).sum(axis=1) / a.sum()
    return vals, gamma(len(cells) + 3) * mag * (1 + 4 * U), mag


def series_prop(vals, step_err, step_mag, first_step, steps_per_period, n):
    """goal_kernel's aligned property of a per-target series [T][1] that carries its own per-step error (an area-weighted mean): the
    period average of the exact steps, with the mean step error added to the kernel's own rounding"""
    T = len(vals)
    depth = 1 + steps_per_period + 1
    val, mag, err = [], [], []
    for i in range(n):
        a = first_step + i * steps_per_period
        idx = range(a, min(a + steps_per_period, T))
        k = len(idx)
        val.append(sum((vals[t] for t in idx), Fraction(0)) / k)
        m = math.fsum(step_mag[t] for t in idx) / k
        mag.append(m)
        err.append((math.fsum(step_err[t] for t in idx) / k + gamma(depth) * m) * (1 + 4 * U))
    return Prop(val, mag, err, [None] * n, np.zeros(n))


def _ieee_class_sum(x):
    """the non-finite value a float64 sum of x gives (NaN if any NaN or both infinities), or None if every term is finite"""
    x = np.asarray(x, dtype=np.float64)
    if np.all(np.isfinite(x)):
        return None
    if np.any(np.isnan(x)) or (np.any(x == np.inf) and np.any(x == -np.inf)):
        return NAN
    return math.inf if np.any(x == np.inf) else -math.inf


def stat_sum_exact(rows, sel, w=None, term_err=None):
    """stat_reduce_rows_kernel: per row sum over the selected cells of w[c] * x[c] (w None: the plain sum), rounded once from the exact
    sum -> (value [R], bound [R]); a row with a non-finite selected term gets the IEEE class of the float sum, bound 0.  term_err [R][n]:
    error bounds of the terms themselves (pot_ratio), added to the bound."""
    X = np.asarray(rows, dtype=np.float64)
    cells = np.flatnonzero(np.asarray(sel, dtype=bool))
    n = X.shape[1]
    wv = np.ones(cells.size) if w is None else np.asarray(w, dtype=np.float64)[cells]
    g = gamma(-(-n // 256) + STAT_TREE + (0 if w is None else 1))
    out, bound = np.zeros(X.shape[0]), np.zeros(X.shape[0])
    for r in range(X.shape[0]):
        x = X[r, cells]
        cls = _ieee_class_sum(x * wv if w is not None else x)
        if cls is not None:
            out[r] = cls
            continue
        out[r], mag = exact_sum(x, wv)
        te = 0.0 if term_err is None else math.fsum(np.asarray(term_err)[r, cells] * np.abs(wv))
        bound[r] = (te + g * (mag + te)) * (1 + 4 * U)
    return out, bound


def pot_ratio_exact(q, area, scale):
    """stat_pot_ratio per cell: 1 - exp(-q / (K area) * 3 / scale) with K the device's float64 m3s_to_mmh constant, exp at 40 digits ->
    (value [..], bound [..]).  The bound allows for the four roundings of the argument (K area, the division, * 3, / scale), one ulp of
    sb_exp (DESIGN.md section 2) and the final subtraction."""
    q = np.asarray(q, dtype=np.float64)
    a = np.broadcast_to(np.asarray(area, dtype=np.float64), q.shape)
    s = np.broadcast_to(np.asarray(scale, dtype=np.float64), q.shape)
    val, bound = np.zeros(q.shape), np.zeros(q.shape)
    with mp.workdps(DPS):
        for ix in np.ndindex(q.shape):
            x = -mpf(float(q[ix])) / (mpf(K_MMH_M3S) * mpf(float(a[ix]))) * 3 / mpf(float(s[ix]))
            e = mp.exp(x)
            val[ix] = float(1 - e)
            ax = abs(float(x))
            bound[ix] = (float(e) * (math.expm1(gamma(4) * ax) + 2 * U) * (1 + gamma(4) * ax + 2 * U) + U * abs(val[ix])) * (1 + 4 * U)
    return val, bound


def ratio(got, want, bound):
    """|got - want| / bound elementwise; 0 where equal, inf where a non-zero error meets a zero bound; a class mismatch of non-finite
    values is inf, a matching class 0"""
    g, w, b = (np.asarray(x, dtype=np.float64).ravel() for x in (got, want, bound))
    out = np.zeros(g.shape)
    for i in range(g.size):
        if not (math.isfinite(w[i]) and math.isfinite(g[i])):
            same = (math.isnan(w[i]) and math.isnan(g[i])) or w[i] == g[i]
            out[i] = 0.0 if same else math.inf
        elif g[i] != w[i]:
            err = abs(math.fsum([g[i], -w[i]])) - 0.5 * math.ulp(w[i])    # want is the exact value rounded once
            out[i] = 0.0 if err <= 0 else (err / b[i] if b[i] > 0 else math.inf)
    return out
