"""The exact interpolation references (tests/interp_reference.py) against the CPU oracle.  The GPU interpolation tests measure the kernels
against these references, so the references are checked first: the oracle is float64 and must land within a few ulps of the
magnitude for IDW and within 1e-12 of max|T| for kriging, which a wrong restatement would not."""
import numpy as np
import pytest

import interp_reference as R
from fixtures import FORCING, geo_matrix

HOUR_US = 3600 * 10**6


def _region(n, T, S, config_index=13, **kw):
    from shyft_b200 import synthetic
    return synthetic.make_region(n, T, S, config_index=config_index, **kw)


def _idw_par(oracle, name):
    return oracle.idw_par(max_members=20 if name in ("temperature", "precipitation") else 10)


@pytest.mark.parametrize("S", [2, 9, 25, 64, 97])
def test_oracle_idw_is_within_a_few_ulps_of_the_exact_mean(oracle, S):
    n, T = 40, 24
    geo, ta, env = _region(n, T, S)
    gm = geo_matrix(geo)
    cells, steps = R.sample_cells(n), R.sample_steps(T)
    for name in FORCING:
        xyz, vals = getattr(env, name)
        vals = oracle.average_accessor_same_axis(vals, HOUR_US)
        par = _idw_par(oracle, name)
        want = oracle.idw_run(name, xyz, vals, gm[:, :3], par, dst_slope=gm[:, 5])[np.ix_(steps, cells)]
        exact, mag = R.idw_exact(oracle, name, xyz, vals, gm[:, :3], par, cells, steps, dst_slope=gm[:, 5])
        err = np.abs(want - exact)
        assert np.all(err <= 16 * R.U * mag), f"S={S} {name}: worst {np.max(err / np.maximum(R.U * mag, 1e-300)):.1f} ulp of the magnitude"


def test_oracle_idw_with_missing_values_and_gradient_by_equation(oracle):
    """NaN station values (reduced neighbour sets) and the 3x3 plane-fit gradient: the fit's round-off is amplified by its condition
    number, so the temperature bound is the oracle's own error there, which must still be small"""
    n, T, S = 40, 24, 25
    geo, ta, env = _region(n, T, S, config_index=12, nan_fraction=0.1)
    gm = geo_matrix(geo)
    cells, steps = R.sample_cells(n), R.sample_steps(T)
    for name in FORCING:
        xyz, vals = getattr(env, name)
        vals = oracle.average_accessor_same_axis(vals, HOUR_US)
        par = oracle.idw_par(max_members=6, gradient_by_equation=True) if name == "temperature" else _idw_par(oracle, name)
        want = oracle.idw_run(name, xyz, vals, gm[:, :3], par, dst_slope=gm[:, 5])[np.ix_(steps, cells)]
        exact, mag = R.idw_exact(oracle, name, xyz, vals, gm[:, :3], par, cells, steps, dst_slope=gm[:, 5])
        assert np.array_equal(np.isnan(want), np.isnan(exact)), name
        ok = ~np.isnan(exact)
        err = np.abs(want - exact)[ok]
        if name == "temperature":
            assert np.max(err) <= 1e-10 * np.max(np.abs(exact[ok])), np.max(err)
        else:
            assert np.all(err <= 16 * R.U * mag[ok]), name


@pytest.mark.parametrize("S", [2, 9, 25, 64, 97])
def test_oracle_btk_is_within_1e_12_of_the_exact_kriging(oracle, S):
    n, T = 40, 12
    geo, ta, env = _region(n, T, S)
    gm = geo_matrix(geo)
    xyz, vals = env.temperature
    vals = oracle.average_accessor_same_axis(vals, HOUR_US)
    cells, steps = R.sample_cells(n), R.sample_steps(T)
    want = oracle.btk_run(xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US)[np.ix_(steps, cells)]
    exact = R.btk_exact(oracle, xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US, cells, steps)
    assert np.max(np.abs(want - exact)) <= 1e-12 * np.max(np.abs(exact))


def test_oracle_btk_on_a_reduced_station_set(oracle):
    n, T, S = 40, 30, 25
    geo, ta, env = _region(n, T, S)
    gm = geo_matrix(geo)
    xyz, vals = env.temperature
    vals = vals.copy()
    vals[8:20, 3] = np.nan
    vals[14:17, [0, 11]] = np.nan
    vals = oracle.average_accessor_same_axis(vals, HOUR_US)
    assert len(R.segments(vals)) == 5
    cells, steps = R.sample_cells(n), R.btk_sample_steps(vals)
    want = oracle.btk_run(xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US)[np.ix_(steps, cells)]
    exact = R.btk_exact(oracle, xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US, cells, steps)
    assert np.max(np.abs(want - exact)) <= 1e-12 * np.max(np.abs(exact))


def test_exact_btk_returns_the_station_value_at_a_station(oracle):
    """a property that does not lean on the oracle: with the covariance's nugget left out of K (sill - nug on the diagonal), a cell on a
    station has k = that column of K, so omega picks the station, BM vanishes and the estimate is the observation itself"""
    S, T = 9, 4
    geo, ta, env = _region(16, T, S)
    xyz, vals = env.temperature
    exact = R.btk_exact(oracle, xyz, vals, xyz[[2, 5]], ta.start * 10**6, HOUR_US, [0, 1], np.arange(T))
    assert np.allclose(exact, vals[:, [2, 5]], rtol=1e-15, atol=0)


def test_samples_cover_the_tile_edges():
    assert list(R.sample_cells(33)) == list(range(33))
    c = R.sample_cells(1030)
    assert len(c) <= 64 and {0, 1029, 127, 128, 1023, 1024}.issubset(set(c))
    assert list(R.sample_steps(9)) == [0, 7, 8]
    assert list(R.sample_steps(65)) == [0, 7, 8, 31, 32, 63, 64]
    v = np.ones((20, 3))
    v[5:12, 1] = np.nan
    assert R.segments(v) == [(0, 5), (5, 12), (12, 20)]
    assert list(R.btk_sample_steps(v)) == [0, 3, 4, 5, 10, 11, 12, 18, 19]
