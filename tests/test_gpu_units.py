"""Device functions one at a time against the oracle (the reference unit-tests its methods the same way:
test/gamma_snow_test.cpp, test/kirchner_test.cpp).  The deterministic math of shyft_b200/csrc/sb2_math.cuh and
oracle/sho_detmath.hpp is one operation sequence written twice: results must be bit-identical."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from shyft_b200 import capi
    return capi


def _bits_equal(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.array_equal(a.view(np.uint64), b.view(np.uint64)) or np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)]) and np.array_equal(np.isnan(a), np.isnan(b))


def test_deterministic_math_is_bit_identical(capi, oracle):
    rng = np.random.default_rng(42)
    x = np.concatenate([rng.uniform(-745, 709, 200000), rng.uniform(-2, 2, 200000), [0.0, -0.0, 1e-300, 709.78, 710.0, -745.0, -746.0, np.nan, np.inf, -np.inf]])
    assert _bits_equal(capi.unit_eval("exp", x)[:, 0], oracle.dm_eval("exp", x))
    x = np.concatenate([np.exp(rng.uniform(-740, 709, 200000)), rng.uniform(0.5, 2.0, 200000), [0.0, 1.0, 5e-324, 1e-310, np.inf, -1.0, np.nan]])
    assert _bits_equal(capi.unit_eval("log", x)[:, 0], oracle.dm_eval("log", x))
    xy = np.stack([rng.uniform(0, 50, 200000), rng.uniform(-4, 4, 200000)], axis=1)
    xy[:8] = [[0, 1.5], [0, -1.5], [2, 0], [3, 1], [3, 2], [9, 0.5], [1.02, 3.5], [5, -1.0 / 3]]
    assert _bits_equal(capi.unit_eval("pow", xy)[:, 0], oracle.dm_eval("pow", xy[:, 0], xy[:, 1]))
    a = rng.uniform(0.05, 60, 200000)
    assert _bits_equal(capi.unit_eval("lgamma", a)[:, 0], oracle.dm_eval("lgamma", a))


def test_branch_free_forms_are_bit_identical(capi, oracle):
    """sb_exp_flat / sb_log_flat / sb_pow_flat (what the production kernels expand in place) against the same oracle functions."""
    rng = np.random.default_rng(43)
    x = np.concatenate([rng.uniform(-745, 709, 200000), rng.uniform(-2, 2, 200000), [0.0, -0.0, 1e-300, 689.9, 690.0, 709.78, 710.0, -745.0, -746.0, np.nan, np.inf, -np.inf]])
    assert _bits_equal(capi.unit_eval("exp_flat", x)[:, 0], oracle.dm_eval("exp", x))
    x = np.concatenate([np.exp(rng.uniform(-740, 709, 200000)), rng.uniform(0.5, 2.0, 200000), [0.0, 1.0, 5e-324, 1e-310, np.inf, -1.0, np.nan]])
    assert _bits_equal(capi.unit_eval("log_flat", x)[:, 0], oracle.dm_eval("log", x))
    xy = np.stack([rng.uniform(0, 50, 200000), rng.uniform(-4, 4, 200000)], axis=1)
    xy[:8] = [[0, 1.5], [0, -1.5], [2, 0], [3, 1], [3, 2], [9, 0.5], [1.02, 3.5], [5, -1.0 / 3]]
    assert _bits_equal(capi.unit_eval("pow_flat", xy)[:, 0], oracle.dm_eval("pow", xy[:, 0], xy[:, 1]))


def test_gamma_p_is_bit_identical_and_accurate(capi, oracle):
    sp = pytest.importorskip("scipy.special")
    rng = np.random.default_rng(7)
    a = rng.uniform(0.1, 8.0, 100000)
    x = rng.uniform(0.0, 1.0, 100000) * (3 * a + 25)
    got = capi.unit_eval("gamma_p", np.stack([a, x], axis=1))[:, 0]
    assert _bits_equal(got, oracle.dm_eval("gamma_p", a, x))
    ref = sp.gammainc(a, x)
    assert np.max(np.abs(got - ref) / np.maximum(ref, 1e-300)) < 5e-13


def test_corr_lwc_known_answer_and_bit_identity(capi, oracle):
    z = capi.unit_eval("corr_lwc", [[4.0, 6.0, 1.0, 5.0, 2.0]])[0, 0]
    assert abs(z - 3.8411) < 1e-4                      # test/gamma_snow_test.cpp:95-108
    rng = np.random.default_rng(11)
    n = 20000
    a1 = rng.uniform(2.0, 6.25, n)
    b1 = rng.uniform(0.05, 8.0, n)
    z1 = rng.uniform(0.01, 1.0, n) * a1 * b1 * 2
    a2 = np.minimum(6.25, a1 * rng.uniform(0.9, 1.2, n))
    b2 = b1 * rng.uniform(1.0, 1.5, n)
    got = capi.unit_eval("corr_lwc", np.stack([z1, a1, b1, a2, b2], axis=1))[:, 0]
    want = np.array([oracle.gs_corr_lwc(z1[i], a1[i], b1[i], 0.0, a2[i], b2[i])[0] for i in range(n)])
    assert _bits_equal(got, want)


def test_calc_snow_state_known_answer_and_bit_identity(capi, oracle):
    swe, sca = capi.unit_eval("calc_snow_state", [[6.25, 0.064, 0.04, 0.0, 0.0, 0.1, 0.0]])[0]
    assert abs(swe - 0.384) < 1e-10 and abs(sca - 0.96) < 1e-10   # test/gamma_snow_test.cpp:76-93
    rng = np.random.default_rng(13)
    n = 20000
    rows = np.stack([rng.uniform(0.1, 6.25, n), rng.uniform(0.0, 20.0, n), np.full(n, 0.04), rng.uniform(-1.0, 60.0, n),
                     rng.uniform(0.0, 30.0, n) * (rng.random(n) < 0.7), np.full(n, 0.1), rng.uniform(0, 2, n) * (rng.random(n) < 0.3)], axis=1)
    rows[:50, 1] = 0.0   # scale 0: lambda/scale = inf takes the bare-ground branch (gamma_snow.h:239-241)
    got = capi.unit_eval("calc_snow_state", rows)
    want = np.array([oracle.gs_calc_snow_state(*r) for r in rows])
    assert _bits_equal(got, want)


def test_kirchner_step_bit_identity_and_known_behaviour(capi, oracle):
    rng = np.random.default_rng(17)
    n = 20000
    q = np.exp(rng.uniform(np.log(1e-6), np.log(60.0), n))
    p = rng.exponential(2.0, n) * (rng.random(n) < 0.5)
    e = rng.uniform(0, 0.3, n)
    rows = np.stack([np.full(n, -2.439), np.full(n, 0.966), np.full(n, -0.10), np.full(n, 1.0), q, p, e], axis=1)
    rows[: n // 4, 3] = 3.0    # 3-hour steps
    rows[n // 4: n // 2, 3] = 24.0
    got = capi.unit_eval("kirchner_step", rows)
    assert np.all(got[:, 2] == 1.0)
    want = np.array([oracle.kirchner_step(r[4], r[5], r[6], dt_us=int(r[3] * 3600 * 10**6))[:2] for r in rows])
    assert _bits_equal(got[:, :2], want)
    # the warp-synchronous solver of the production kernels: lanes with 1..n sub-steps share a warp, n not a multiple of 32
    rows_w = rows[: n - 7]
    got_w = capi.unit_eval("kirchner_step_warp", rows_w)
    assert np.all(got_w[:, 2] == 1.0)
    assert _bits_equal(got_w[:, :2], want[: n - 7])
    # P = 10, E = 0 from q = 1: q and q_avg converge to 10 (test/kirchner_test.cpp:40-54)
    row = np.array([[-2.439, 0.966, -0.10, 1.0, 1.0, 10.0, 0.0]])
    for _ in range(3000):
        out = capi.unit_eval("kirchner_step", row)
        row[0, 4] = out[0, 0]
    assert abs(out[0, 0] - 10.0) < 1e-3 and abs(out[0, 1] - 10.0) < 1e-3


def test_division_by_a_step_invariant_divisor_is_the_ieee_quotient(capi):
    """div_by (sb2_math.cuh): a / d through the once-divided reciprocal and two fused corrections -- Markstein's theorem makes it the
    correctly rounded quotient; the out-of-range numerators and divisors take the IEEE division.  Bit for bit against a / d on the
    device and on the host."""
    rng = np.random.default_rng(23)
    n = 2_000_000
    a = rng.standard_normal(n) * np.exp(rng.uniform(-40, 40, n))
    d = np.exp(rng.uniform(-12, 24, n))
    # the divisors of the step kernels, zero / tiny / huge / non-finite numerators, divisors with all-ones and all-zeros mantissas
    d[:9] = [3600000000.0, 3600.0, 333660.0, 5.0, 0.96, 0.1, 0.16, 1.5, 0.4 * 0.4]
    a[:64:7] = 0.0
    a[1:64:7] = -0.0
    a[100:110] = [np.inf, -np.inf, np.nan, 5e-324, 1e-310, 1e-250, 1e250, 1.7e308, -1e-300, 2.0**-823]
    d[200:300] = np.nextafter(2.0 ** rng.integers(-20, 20, 100).astype(np.float64), 0.0)
    d[300:400] = 2.0 ** rng.integers(-20, 20, 100).astype(np.float64)
    d[400:410] = [0.0, np.inf, np.nan, 1e-300, 1e300, -3.0, -0.5, 2.0**-200, 2.0**199, 5e-324]
    got = capi.unit_eval("div_by", np.stack([a, d], axis=1))
    with np.errstate(all="ignore"):
        want = a / d
    assert _bits_equal(got[:, 1], want)          # the device's own IEEE division
    assert _bits_equal(got[:, 0], want)          # div_by


def test_kirchner_first_try_with_host_evaluated_products_is_bit_identical(capi, oracle):
    """kirchner_step_warp<true>: the first try of a step multiplies the slopes with dt * tableau products evaluated on the host (the
    production kernels' form) -- same bits as the per-lane products, with 1..n sub-step lanes mixed in a warp"""
    rng = np.random.default_rng(19)
    n = 20000 - 5
    q = np.exp(rng.uniform(np.log(1e-6), np.log(60.0), n))
    p = rng.exponential(2.0, n) * (rng.random(n) < 0.5)
    p[::50] *= 40.0                                  # cloudbursts: rejected first tries, several sub-steps
    e = rng.uniform(0, 0.3, n)
    rows = np.stack([np.full(n, -2.439), np.full(n, 0.966), np.full(n, -0.10), np.full(n, 1.0), q, p, e], axis=1)
    got = capi.unit_eval("kirchner_step_warp_udt", rows)
    assert np.all(got[:, 2] == 1.0)
    want = np.array([oracle.kirchner_step(r[4], r[5], r[6])[:2] for r in rows])
    assert _bits_equal(got[:, :2], want)
    assert _bits_equal(capi.unit_eval("kirchner_step_warp", rows)[:, :2], want)


def test_kirchner_first_try_out_of_the_fast_exp_range(capi, oracle):
    """The first try defers arguments outside exp's fast range (|.| >= 690) to a repeat of the whole try with the full-range exp: warps that
    mix such lanes (c1 around -700: g(q) underflows, the response is frozen) with ordinary ones give the oracle's bits on every lane.
    (Only the underflow side: an overflowing g sends the reference's own controller into millions of sub-steps.)"""
    rng = np.random.default_rng(23)
    n = 32 * 32
    q = np.exp(rng.uniform(np.log(1e-6), np.log(60.0), n))
    p = rng.exponential(2.0, n) * (rng.random(n) < 0.5)
    e = rng.uniform(0, 0.3, n)
    c = np.tile(np.array([-2.439, 0.966, -0.10]), (n, 1))
    wild = rng.random(n) < 0.2
    wild[:32] = False                                # one warp without any, the rest mixed
    c[wild] = np.stack([rng.uniform(-760, -690, wild.sum()), rng.uniform(-1, 1, wild.sum()), rng.uniform(-0.2, 0.2, wild.sum())], axis=1)
    rows = np.concatenate([c, np.ones((n, 1)), q[:, None], p[:, None], e[:, None]], axis=1)
    got = capi.unit_eval("kirchner_step_warp_udt", rows)
    want = np.array([oracle.kirchner_step(q[i], p[i], e[i], c=tuple(c[i]))[:2] for i in range(n)])
    assert wild.sum() > 100 and np.all(got[:, 2] == 1.0)
    assert _bits_equal(got[:, :2], want)
    assert _bits_equal(capi.unit_eval("kirchner_step_warp", rows)[:, :2], want)
