"""The routing references of routing_reference.py against independent arithmetic, and the library's and the oracle's gamma unit
hydrographs and river flows against them (no GPU needed).  The GPU routing tests compare the kernels with the oracle, so the oracle is
checked here first."""
import math

import numpy as np
import pytest
from mpmath import mp

import routing_reference as R

ALPHAS = (0.3, 0.6, 1.0, 1.5, 3.0, 7.0, 20.0, 80.0)
BETAS = (0.0, 0.1, -0.02, -1.0e3)                # -1e3 is below every pdf value of the grid: all taps zero, the 1/n fallback
STEPS = (2, 3, 7, 24, 64, 137, 500)
# Both float64 implementations solve P(alpha, x_max) = 0.99 by Newton to |dx| <= 1e-15 x and evaluate the pdf at x <= x_max as
# exp((alpha - 1) log x - x - lgamma(alpha)), exp and log within 1.5 ulp.  The relative error of a tap is then at most
#   - the exponent's rounding: log x, the product, the difference and exp each within 2u of the largest term, |alpha - 1| |log x| or x,
#     doubled for the normalisation and the comparison with max w: 8u (|alpha - 1| |log x_max| + x_max);
#   - the quantile's: a relative error eps of x_max moves pdf(x) by |alpha - 1 - x| eps <= (|alpha - 1| + x_max) 1e-15.
# lgamma(alpha) is shared by all taps and cancels in the normalisation; +beta does not cancel, but the pdf terms bound it.  This is
# 6e-15 of max w at alpha = 0.3, 1.2e-13 at 20 and 5.9e-13 at 80; the worst measured over the grid are 1.8e-15, 1.45e-14 and 2.0e-13.
def uhg_tol(alpha):
    x = float(R.gamma_quantile_exact(alpha))
    return 8 * R.U * (abs(alpha - 1) * abs(math.log(x)) + x) + 1e-15 * (abs(alpha - 1) + x)


WORST = {}


@pytest.fixture(scope="module")
def capi():
    from shyft_b200 import capi as c
    return c


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nworst unit-hydrograph error against the 40-digit reference, as a fraction of its bound: " + ", ".join(f"{k} {v:.2f}" for k, v in WORST.items()))


def _host_uhg(capi, n, alpha, beta):
    got = capi.host_eval(2, [n, alpha, beta], 1001)
    return got[1:1 + int(got[0])]


@pytest.mark.parametrize("alpha", ALPHAS)
def test_unit_hydrographs_against_the_exact_gamma(capi, oracle, alpha):
    for beta in BETAS:
        for n in STEPS:
            want = np.array([float(v) for v in R.uhg_exact(n, alpha, beta)])
            assert want.size == n and abs(want.sum() - 1.0) < 1e-15
            for name, got in (("host", _host_uhg(capi, n, alpha, beta)), ("oracle", oracle.make_uhg(n, alpha, beta))):
                assert got.size == n, (name, n, alpha, beta)
                assert np.array_equal(got == 0, want == 0), (name, n, alpha, beta)    # +beta truncation at the same taps
                err = np.max(np.abs(got - want)) / np.max(want)
                WORST[name] = max(WORST.get(name, 0.0), err / uhg_tol(alpha))
                assert err <= uhg_tol(alpha), f"{name} n={n} alpha={alpha} beta={beta}: {err:.2e} of max w"
    if alpha == 1.0:
        assert np.array_equal(_host_uhg(capi, 5, 1.0, -1e3), np.full(5, 0.2))
    for n in (0, 1):
        assert [float(v) for v in R.uhg_exact(n, alpha, 0.0)] == [1.0] and _host_uhg(capi, n, alpha, 0.0).tolist() == [1.0]


def test_the_quantile_is_the_gamma_quantile():
    """x_max against an independent identity: for alpha = 1 P(1, x) = 1 - exp(-x), so x = ln 100"""
    with mp.workdps(40):
        assert abs(R.gamma_quantile_exact(1.0) - mp.log(100)) < mp.mpf(10) ** -35
        assert abs(mp.gammainc(20, 0, R.gamma_quantile_exact(20.0), regularized=True) - mp.mpf("0.99")) < mp.mpf(10) ** -35


def test_exact_sum_is_the_40_digit_sum():
    """exact_sum (two-product + fsum) equals the 40-digit mpmath dot product rounded to float64, also under heavy cancellation"""
    rng = np.random.default_rng(5)
    for k in range(20):
        a = rng.uniform(0, 1, 500) * 10.0 ** rng.integers(-30, 3, 500)
        b = rng.normal(0, 1, 500) * 10.0 ** rng.integers(-3, 3, 500)
        if k % 2:
            b[250:] = -b[:250] * a[:250] / a[250:]                  # terms that nearly cancel in pairs
        with mp.workdps(40):
            want = float(mp.fdot(a.tolist(), b.tolist()))
        got, mag = R.exact_sum(a, b)
        assert got == want, k
        assert mag == pytest.approx(np.sum(np.abs(a * b)), rel=1e-13)


def tree_case():
    """a small branching network with multi-tap unit hydrographs: rivers in shuffled id order, fan-in 3 into river 4, a chain 7 -> 2
    -> 4, river 6 without cells, unrouted cells in between; hourly steps"""
    rivers = np.array([[2, 4, 3.0 * 3600, 1.0, 3.0, 0.0], [7, 2, 5.0 * 3600, 1.0, 0.6, 0.1], [4, 0, 9.0 * 3600, 1.0, 7.0, 0.0],
                       [1, 4, 1.0 * 3600, 1.0, 7.0, 0.0], [6, 4, 12.0 * 3600, 2.0, 1.5, -0.02], [3, 7, 0.0, 1.0, 7.0, 0.0]])
    rng = np.random.default_rng(11)
    n, T = 60, 90
    rid = rng.choice([0, 1, 2, 3, 4, 7], n)
    dist = rng.choice([0.0, 3600.0, 7200.0, 24 * 3600.0, 30 * 3600.0], n)
    par = np.stack([rng.choice([0.5, 1.0, 2.0], n), rng.choice([0.6, 3.0, 7.0], n), rng.choice([0.0, 0.1, -0.02], n)], axis=1)
    q = rng.exponential(2.0, (T, n))
    return rivers, q, rid.astype(np.int64), dist, par


def test_oracle_river_flows_against_the_exact_network(capi, oracle):
    """every river of tree_case, every step: each stage of the oracle from its own inputs against the exact sum, within the float64
    bound of the oracle's summation order (per cell: L taps, then n_cells into local; n_up into upstream, +1, L taps into output)"""
    rivers, q, rid, dist, par = tree_case()
    T = q.shape[0]
    steps = np.arange(T)
    flows = {int(r): oracle.river_flows(rivers, int(r), q, rid, dist, par, 3600 * 10**6) for r in rivers[:, 0]}
    w_cell = [_host_uhg(capi, int(capi.host_eval(3, [dist[c], par[c, 0], 3600 * 10**6], 1)[0]), par[c, 1], par[c, 2]) for c in range(len(rid))]
    for r, down, d, v, a, b in rivers:
        r = int(r)
        local, up, out = flows[r]
        cells = np.flatnonzero(rid == r)
        lx, lmag = R.local_exact(q, cells, w_cell, steps)
        L = max((len(w_cell[c]) for c in cells), default=1)
        assert np.all(np.abs(local - lx) <= (L + len(cells) + 1) * R.U * lmag), r
        ups = [int(u) for u in sorted(rivers[rivers[:, 1] == r, 0])]
        w = _host_uhg(capi, int(capi.host_eval(3, [d, v, 3600 * 10**6], 1)[0]), a, b)
        assert np.array_equal(w, oracle.make_uhg(len(w), a, b)) or np.allclose(w, oracle.make_uhg(len(w), a, b), rtol=0, atol=uhg_tol(a))
        ux, umag, ox, omag = R.river_exact(local, [flows[u][2] for u in ups], oracle.make_uhg(len(w), a, b), steps)
        assert np.all(np.abs(up - ux) <= max(len(ups), 1) * R.U * umag), r
        assert np.all(np.abs(out - ox) <= (len(w) + len(ups) + 1) * R.U * omag), r
    assert len(np.flatnonzero(rid == 6)) == 0 and flows[6][0].max() == 0.0 and flows[6][2].max() == 0.0
    assert flows[4][1].max() > 0 and len(rivers[rivers[:, 1] == 4]) == 3
