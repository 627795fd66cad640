"""The statistics reduction kernels (shyft_b200/csrc/sb2_stats.cuh) against the exact references of tests/goal_reference.py.

The forcing readers read the resident cell environment, so the values are set directly (initialize_cell_environment + set_cell_forcing)
and nothing is run: cells in {1, 31, 32, 33, 255, 256, 257, 5 000} around the warp and the 256-thread block, rows in {1, 1 184, 1 185,
3 000} around the 1 184-block grid of stat_reduce_rows_kernel, whose blocks then reduce a second row; selections of all cells, one
catchment, interleaved catchments and scattered, unsorted cell lists with duplicates; values of mixed sign with heavy cancellation, over
1e-300 .. 1e290 (clear of overflow with areas up to 1e8 m2), and NaN / +-inf in selected and in unselected cells (which must not leak).
Readers: the area average (temperature), the area-average value (temperature_value, / sum_area on the host), the gather (temperature(sel,
step)) and the plain sum (w = null), and the three forms of pot_ratio on a short pt_hs_k run.  Finite sums are held to the exact sum within
gamma(strides + 13) of the magnitude; a non-finite row must have the IEEE class of the float64 sum."""
import time

import numpy as np
import pytest

import goal_reference as G

pytestmark = pytest.mark.gpu
GRID = 148 * 8                       # stat_reduce_rows_kernel: at most 1 184 blocks
START = 1420070400
WORST = {}


def note(case, r):
    WORST[case] = max(WORST.get(case, 0.0), float(np.max(r)) if np.size(r) else 0.0)


@pytest.fixture(scope="module", autouse=True)
def _report():
    t0 = time.perf_counter()
    yield
    print("\nworst statistics error per case, in units of its exact bound (<= 1 passes):")
    for case, r in sorted(WORST.items()):
        print(f"  {case:44s} {r:.3e}")
    print(f"module wall time {time.perf_counter() - t0:.1f} s")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def values(rows, n, seed):
    """row r % 4: 0 wide range, 1 heavy cancellation, 2 non-finite values in cells 2 and n-1 (unselected by the catchment selections),
    3 non-finite in cells 0 and 1 (selected by every selection but catchment 2's)"""
    rng = np.random.default_rng(seed)
    X = rng.choice([-1.0, 1.0], (rows, n)) * 10.0 ** rng.uniform(-300, 290, (rows, n))
    big = rng.normal(0, 1, (rows, n)) * 1e12
    canc = big.copy()
    canc[:, 1::2] = -canc[:, 0::2][:, : n // 2] * (1 + rng.normal(0, 1e-9, (rows, n // 2)))
    kind = np.arange(rows) % 4
    X[kind == 1] = canc[kind == 1] + rng.normal(0, 1, (rows, n))[kind == 1]
    bad = [np.nan, np.inf, -np.inf]
    for r in np.flatnonzero(kind >= 2):
        c0, c1 = (2 % n, n - 1) if kind[r] == 2 else (0, 1 % n)
        X[r, c0] = bad[(r // 4) % 3]
        if (r // 4) % 5 == 4:
            X[r, c1] = np.inf if X[r, c0] == -np.inf else -np.inf
    return X


def region(sb, n, rows, seed):
    """n cells in catchments 1 (cells 0, 1 and every 3rd), 2 and 3, areas over 1e3 .. 1e8 m2; the temperature set to values()"""
    from shyft_b200 import synthetic
    rng = np.random.default_rng(seed)
    geo = synthetic.make_cells(n, rng)[0]
    geo["area"] = 10 ** rng.uniform(3, 8, n)
    cid = 1 + np.arange(n) % 3
    cid[:2] = 1
    cid[2 % n] = 2 if n > 2 else 1
    cid[n - 1] = 2 if n > 2 else 1
    geo["catchment_id"] = cid
    m = sb.PTGSKModel(geo)
    m.initialize_cell_environment(sb.TimeAxis(START, 3600, rows))
    X = values(rows, n, seed)
    m.set_cell_forcing("temperature", X)
    return m, X, np.asarray(geo["area"]), cid


def selections(n, cid):
    from shyft_b200.statistics import CATCHMENT_IX, CELL_IX
    rng = np.random.default_rng(n)
    scattered = list(rng.integers(0, n, max(3, n // 3))) + [0, 0, n - 1]
    rng.shuffle(scattered)
    out = {"all": ([], CATCHMENT_IX, np.ones(n, dtype=bool)), "one catchment": ([1], CATCHMENT_IX, cid == 1),
           "cells scattered, duplicated": ([int(x) for x in scattered], CELL_IX, np.isin(np.arange(n), scattered))}
    if 2 in cid and 3 in cid:
        out["catchments 3, 1 interleaved"] = ([3, 1], CATCHMENT_IX, np.isin(cid, [1, 3]))
    return out


SHAPES = [(1, 1185), (31, 1), (32, 1184), (33, 1185), (255, 3000), (256, 1), (257, 1184), (5000, 1185)]


@pytest.mark.parametrize("shape", SHAPES, ids=[f"{n}cells_{r}rows" for n, r in SHAPES])
def test_forcing_readers_against_exact_sums(sb, shape):
    from test_gpu_step_paths import launched
    n, rows = shape
    m, X, area, cid = region(sb, n, rows, seed=n + rows)
    assert np.array_equal(m.cell_forcing("temperature"), X, equal_nan=True)
    steps = sorted({0, rows // 2, rows - 1})
    for name, (idx, ix, sel) in selections(n, cid).items():
        case = f"{n} cells x {rows} rows, {name}"
        # the plain sum (kind forcing, op sum)
        got = []
        ks = launched(lambda: got.append(m.statistics._series(0, 0, idx, ix, 0)))
        want, bound = G.stat_sum_exact(X, sel)
        r = G.ratio(got[0], want, bound)
        note("sum " + case.split(",")[0], r)
        assert np.all(r <= 1.0), (case, "sum", np.flatnonzero(r > 1)[:5], got[0][r > 1][:5], want[r > 1][:5])
        grids = [g for k, g in ks if k == "stat_reduce_rows_kernel"]
        assert len(grids) == 1 and grids[0][0] == min(rows, GRID), (case, ks)
        # the area average: r * (1 / sum_area) on the host, and the value form r / sum_area
        wsum, wbound = G.stat_sum_exact(X, sel, area)
        sa = float(np.sum(area[sel]))
        avg, avb = wsum / sa, wbound / sa + G.gamma(int(sel.sum()) + 2) * np.abs(wsum / sa)
        got = m.statistics.temperature(idx, ix_type=ix)
        r = G.ratio(got, avg, avb)
        note("area average " + case.split(",")[0], r)
        assert np.all(r <= 1.0), (case, "average", np.flatnonzero(r > 1)[:5])
        for j in steps:
            r = G.ratio(m.statistics.temperature_value(idx, j, ix_type=ix), avg[j], avb[j])
            note("area average value " + case.split(",")[0], r)
            assert np.all(r <= 1.0), (case, "value", j)
            assert np.array_equal(m.statistics.temperature(idx, j, ix_type=ix), X[j, np.flatnonzero(sel)], equal_nan=True), (case, j)
    # a row with non-finite values only in unselected cells stays finite: every selection above that leaves cells 2 and n-1 out
    if n > 3:
        r2 = np.flatnonzero(np.arange(rows) % 4 == 2)
        if r2.size:
            assert np.all(np.isfinite(m.statistics.temperature([1], ix_type=0)[r2]))


def test_pot_ratio_forms(sb):
    """pot_ratio = 1 - exp(-m3s_to_mmh(kirchner_discharge) * 3 / ae_scale) per cell: its sum, area average and gather"""
    from fixtures import PTHSK_DEFAULT
    from shyft_b200 import synthetic
    from shyft_b200.statistics import CELL_IX
    n, T = 257, 240
    geo, ta, env = synthetic.make_region(n, T, 4, config_index=44, cells_per_catchment=90, start=START)
    geo["area"] = 10 ** np.random.default_rng(6).uniform(3, 8, n)
    m = sb.PTHSKModel(geo, PTHSK_DEFAULT)
    assert m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(synthetic.default_state(1, n))
    m.set_state_collection(-1, True)
    m.run_cells()
    kd = m.state_series("kirchner_discharge")
    area = np.asarray(geo["area"])
    pr, pb = G.pot_ratio_exact(kd, area[None, :], PTHSK_DEFAULT[3])
    cid = np.asarray(geo["catchment_id"])
    for idx, ix, sel in (([], 0, np.ones(n, dtype=bool)), ([2], 0, cid == 2), ([5, 250, 5, 0, 128], CELL_IX, np.isin(np.arange(n), [0, 5, 128, 250]))):
        got = m.statistics._series(3, 0, idx, ix, 0)
        want, bound = G.stat_sum_exact(pr, sel, term_err=pb)
        r = G.ratio(got, want, bound)
        note("pot_ratio sum", r)
        assert np.all(r <= 1.0), ("sum", idx)
        wsum, wbound = G.stat_sum_exact(pr, sel, area, term_err=pb)
        sa = float(np.sum(area[sel]))
        got = m.actual_evaptranspiration_response.pot_ratio(idx, ix_type=ix)
        r = G.ratio(got, wsum / sa, wbound / sa + G.gamma(int(sel.sum()) + 2) * np.abs(wsum / sa))
        note("pot_ratio area average", r)
        assert np.all(r <= 1.0), ("average", idx)
        for j in (0, 120, T):
            got = m.actual_evaptranspiration_response.pot_ratio(idx, j, ix_type=ix)
            r = G.ratio(got, pr[j, sel], pb[j, sel])
            note("pot_ratio gather", r)
            assert np.all(r <= 1.0), ("gather", idx, j)
