"""Exact references of routing: the gamma unit hydrograph in mpmath at 40 significant digits, and the three flows of a river.

uhg_exact restates make_uhg_from_gamma (core/routing.h:399-421) with mpmath's regularised incomplete gamma and gamma function in place
of boost::math::gamma_distribution.  The flows restate routing::model (core/routing.h:326-383) with the USE_ZERO convolution of
core/time_series.h:966-975, one stage at a time and from the inputs a device hands that stage: local inflow from cell discharge,
upstream inflow and output from the device's own local inflow and upstream outputs.  So each kernel is measured against its own
operation, and errors do not compound from stage to stage.

A flow is a sum of products of float64 numbers.  exact_sum forms every product exactly (Dekker's two-product: p + e = a * b with no
rounding) and adds them with math.fsum, which returns the exact sum rounded once: within half an ulp of the true value, the same as a
40-digit mpmath sum rounded to float64, and much faster on the 10^5-term sums of a 300-cell river (test_routing_reference_cpu checks
the two agree).  Every result comes with its magnitude, the sum of the absolute values of its terms.
"""
import math

import numpy as np
from mpmath import mp, mpf

DPS = 40
U = 2.0**-53                 # unit round-off of float64
_SPLIT = 134217729.0         # 2^27 + 1 (Veltkamp)


_QUANTILE = {}


def gamma_quantile_exact(alpha):
    """x with P(alpha, x) = 0.99 (regularised lower incomplete gamma), to 40 digits: bracketed, then solved by findroot"""
    if alpha not in _QUANTILE:
        with mp.workdps(DPS):
            a = mpf(alpha)
            p = lambda x: mp.gammainc(a, 0, x, regularized=True) - mpf("0.99")
            hi = max(mpf(1), a)
            while p(hi) < 0:
                hi *= 2
            _QUANTILE[alpha] = mp.findroot(p, (hi / 2 if p(hi / 2) < 0 else mpf(0), hi), solver="illinois")
    return _QUANTILE[alpha]


def uhg_exact(n_steps, alpha, beta):
    """make_uhg_from_gamma at 40 digits -> list of mpf: x_max solves P(alpha, x) = 0.99, tap i = max(0, pdf(i * x_max / n) + beta),
    pdf(0) = 0 for every shape (boost 1.68), normalised; all taps zero -> 1/n each; n <= 1 -> [1]"""
    with mp.workdps(DPS):
        if n_steps <= 1:
            return [mpf(1)]
        a, b = mpf(alpha), mpf(beta)
        d = gamma_quantile_exact(alpha) / n_steps
        pdf = lambda x: mpf(0) if x == 0 else mp.exp((a - 1) * mp.log(x) - x - mp.loggamma(a))
        y = [max(mpf(0), pdf(d * i) + b) for i in range(n_steps)]
        s = mp.fsum(y)
        return [v / s for v in y] if s > 0 else [mpf(1) / n_steps] * n_steps


def _two_product(a, b):
    """p + e == a * b exactly (no overflow or underflow at the magnitudes of discharge and unit-hydrograph weights)"""
    p = a * b
    ca, cb = _SPLIT * a, _SPLIT * b
    ah, bh = ca - (ca - a), cb - (cb - b)
    al, bl = a - ah, b - bh
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def exact_sum(a, b):
    """sum a[i] * b[i] rounded once, and sum |a[i] * b[i]|"""
    a, b = np.asarray(a, dtype=np.float64).ravel(), np.asarray(b, dtype=np.float64).ravel()
    p, e = _two_product(a, b)
    return math.fsum(np.concatenate([p, e])), math.fsum(np.abs(p))


def _convolve(series, w, t):
    """sum_j w[j] * series[t - j] over j <= t as (weights, values): series [T][k], w [L] -> flattened term pairs"""
    j = np.arange(min(len(w), t + 1))
    vals = series[t - j]                                        # [len(j)][k]
    return np.repeat(np.asarray(w)[j], vals.shape[1] if vals.ndim > 1 else 1), vals.ravel()


def local_exact(q, cells, weights, steps):
    """local inflow of a river: q [T][n_cells] device cell discharge, cells = the river's cell indices, weights[c] = the cell's unit
    hydrograph (float64, as the library builds it) -> (value [len(steps)], magnitude [len(steps)])"""
    val, mag = np.zeros(len(steps)), np.zeros(len(steps))
    by_w = {}
    for c in cells:                                             # cells with the same unit hydrograph convolve together
        by_w.setdefault(tuple(weights[c]), []).append(c)
    for k, t in enumerate(steps):
        wa, va = [], []
        for w, cs in by_w.items():
            a, b = _convolve(q[:, cs], w, t)
            wa.append(a)
            va.append(b)
        val[k], mag[k] = exact_sum(np.concatenate(wa), np.concatenate(va)) if wa else (0.0, 0.0)
    return val, mag


def river_exact(local, ups, w, steps):
    """upstream inflow and output of a river from the device's local inflow [T] and upstream outputs (list of [T]), w = the river's
    unit hydrograph -> (upstream, upstream magnitude, output, output magnitude), each [len(steps)]"""
    src = np.stack([local] + list(ups), axis=1)                 # [T][1 + n_up]
    up, up_mag, out, out_mag = (np.zeros(len(steps)) for _ in range(4))
    for k, t in enumerate(steps):
        if ups:
            up[k], up_mag[k] = exact_sum(np.ones(len(ups)), src[t, 1:])
        out[k], out_mag[k] = exact_sum(*_convolve(src, w, t))
    return up, up_mag, out, out_mag


def sample_steps(T, window_edges=(), n_random=64, seed=0):
    """0, 63, 64, 65, 127, 128 and T-1 (the 64-step time tiles of both kernels), the given window edges and both sides of them, and
    n_random random steps"""
    picks = {0, 63, 64, 65, 127, 128, T - 1}
    for e in window_edges:
        picks.update((e - 1, e))
    rng = np.random.default_rng(seed)
    picks.update(rng.integers(0, T, min(n_random, T)).tolist())
    return np.array(sorted(s for s in picks if 0 <= s < T), dtype=np.int64)
