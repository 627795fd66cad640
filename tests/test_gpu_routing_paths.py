"""Both routing kernels and the river network, against the CPU oracle and against the exact references of routing_reference.py.

route_local_inflow_kernel (shyft_b200/csrc/sb2_routing.cuh) convolves each cell's discharge with its unit hydrograph (UHG) over a
64-step tile, 128 cells a chunk, one lane per cell and a 5-level shuffle tree per warp; route_river_level_kernel convolves the sum of a
river's local inflow and its upstream rivers' outputs with the river's UHG, one network level a launch.  Cell discharge comes from a
short hbv_stack run and is read back from the device, so routing is measured apart from the step kernels.

Cases ("taps" = UHG length; cell taps are set through routing_distance and per-catchment routing velocity / alpha / beta):

    case         T    dt s    network                                   cells per river            cell taps            river taps
    fan3_mixed   65   3600    1, 2, 3 -> 4; 4, 6 -> 5; shuffled ids     1, 31, 128, 129, 300, 0    2, 24, 1, 64/65/2/24  1, 64, 200, 65, 3, 3
                              river 6 without cells, 20 unrouted cells  (129: three catchments in one warp, one with beta < 0)  (300: 137)
    tree5_15min  999  900     binary tree of 5 uneven levels,           300 (3 chunks), 1..40      1, 2, 24             1, 3, 64, 65, 1000
                              ids listed in descending order                                                             (1000 > T)
    t1_3h        1    10800   2 -> 1                                    31, 1                      2, 1                 3, 1
    t63          63   900     1 -> 2, 3 -> 2                            129, 1, 31                 65, 1, 24            64, 1, 3
    t64          64   3600    2 -> 1                                    128, 129                   64, 137              65, 200

Every river of every case is checked (a) against oracle.river_flows over all steps at rtol 1e-12; (b) against the exact reference on the
sample of routing_reference.sample_steps (0, 63, 64, 65, 127, 128, T-1 and 64 random steps): local inflow within
K = L_cell + ceil(n_chunk_cells / 32) + 5 + n_chunks times 2^-53 of its magnitude (the sequential tap sum, a lane's cells, the shuffle tree,
the chunk accumulation), upstream inflow and output within K = L_river + n_up + 1.  The worst errors per kernel and case are printed at
the end of the module.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import routing_reference as R
from fixtures import HBV_DEFAULT
from parity import parity_report

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-12
ROUTE = slice(17, 20)                    # routing velocity, alpha, beta in the hbv_stack parameter vector
MIXED = {11: (1.0, 3.0, 0.0), 12: (0.5, 0.6, -0.02), 13: (2.0, 20.0, 0.1)}

# name: T, dt, rivers [(id, downstream id, taps, velocity, alpha, beta)], cell groups [(river id, count, catchment id(s), taps)],
# catchment routing parameters {cid: (velocity, alpha, beta)}
CASES = {
    "fan3_mixed": (65, 3600, [(3, 4, 200, 1.0, 3.0, 0.0), (5, 0, 3, 1.0, 7.0, 0.0), (1, 4, 1, 1.0, 7.0, 0.0), (6, 5, 3, 2.0, 0.6, 0.1),
                              (4, 5, 65, 0.5, 1.5, -0.02), (2, 4, 64, 1.0, 7.0, 0.0)],
                   [(1, 1, 1, 2), (2, 31, 2, 24), (3, 128, 3, 1), (4, 129, (11, 12, 13), (64, 65, 2, 24)), (5, 300, 5, 137), (0, 20, 9, 3)],
                   MIXED),
    "tree5_15min": (999, 900, [(9, 0, 1000, 1.0, 7.0, 0.0), (8, 9, 65, 1.0, 3.0, 0.0), (7, 9, 1, 1.0, 7.0, 0.0), (6, 8, 64, 1.0, 7.0, 0.0),
                               (5, 8, 3, 1.0, 7.0, 0.0), (4, 6, 3, 1.0, 0.6, 0.0), (3, 6, 1, 1.0, 7.0, 0.0), (2, 4, 64, 2.0, 20.0, 0.0),
                               (1, 4, 3, 1.0, 7.0, 0.0)],
                    [(9, 40, 1, 24), (8, 300, (11, 12, 13), (2, 24, 1)), (7, 1, 1, 2), (6, 31, 1, 1), (5, 33, 12, 24), (4, 7, 1, 2),
                     (3, 1, 13, 24), (2, 129, 1, 2), (1, 5, 1, 24), (0, 9, 1, 2)], MIXED),
    "t1_3h": (1, 10800, [(2, 1, 3, 1.0, 7.0, 0.0), (1, 0, 1, 1.0, 7.0, 0.0)], [(2, 31, 1, 2), (1, 1, 1, 1)], {}),
    "t63": (63, 900, [(1, 2, 64, 1.0, 7.0, 0.0), (2, 0, 1, 1.0, 7.0, 0.0), (3, 2, 3, 1.0, 7.0, 0.0)],
            [(1, 129, (11, 12), 65), (2, 1, 1, 1), (3, 31, 13, 24)], MIXED),
    "t64": (64, 3600, [(2, 1, 65, 1.0, 7.0, 0.0), (1, 0, 200, 1.0, 0.6, 0.1)], [(2, 128, 1, 64), (1, 129, 1, 137)], {}),
}

WORST = {}   # (kernel, case) -> {"oracle": max|got - want| / max|want|, "exact": worst error in ulps of the magnitude}


def _note(key, what, value):
    d = WORST.setdefault(key, {})
    d[what] = max(d.get(what, 0.0), float(value))


def _worst_table():
    return "; ".join(f"{k[0]} {k[1]}: oracle {v.get('oracle', 0):.2e}, exact {v.get('exact', 0):.2f} ulps" for k, v in sorted(WORST.items()))


@pytest.fixture(scope="module", autouse=True)
def _report_worst_errors():
    yield
    print("\nworst errors per kernel and case (oracle: max|got - want| / max|want|; exact: in 2^-53 of the magnitude)")
    for (k, c), v in sorted(WORST.items()):
        print(f"  {k:12s} {c:14s} oracle {v.get('oracle', 0):.3e}   exact {v.get('exact', 0):7.2f} ulps")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


# ---- set-up -------------------------------------------------------------------------------------------------------------------------
def catchment_parameter(vel_alpha_beta, base=HBV_DEFAULT):
    p = np.array(base, dtype=np.float64)
    p[ROUTE] = vel_alpha_beta
    return p


class Region:
    """a case laid out as cells: routing ids interleaved (shuffled with a fixed seed), distances that give each cell its taps"""

    def __init__(self, T, dt, rivers, groups, catch, seed=7, region_route=None):
        from shyft_b200 import synthetic
        self.T, self.dt, self.catch = T, dt, dict(catch)
        self.region_route = tuple(HBV_DEFAULT[ROUTE]) if region_route is None else region_route
        spec = []
        for rid, count, cid, taps in groups:
            cids = cid if isinstance(cid, tuple) else (cid,)
            tl = taps if isinstance(taps, tuple) else (taps,)
            spec += [(rid, cids[k % len(cids)], tl[k % len(tl)]) for k in range(count)]
        spec = [spec[i] for i in np.random.default_rng(seed).permutation(len(spec))]
        self.n = len(spec)
        geo, self.ta, self.env = synthetic.make_region(self.n, T, 4, config_index=seed, dt=dt, with_routing=True)
        self.geo = geo.copy()
        self.rid = np.array([s[0] for s in spec], dtype=np.int64)
        self.cid = np.array([s[1] for s in spec], dtype=np.int64)
        self.taps = np.array([s[2] for s in spec])
        self.geo["routing_id"] = self.rid
        self.geo["catchment_id"] = self.cid
        self.geo["routing_distance"] = self.taps * self.cell_par()[:, 0] * dt
        self.rivers = np.array([[r, d, taps * v * dt, v, a, b] for r, d, taps, v, a, b in rivers], dtype=np.float64)

    def cell_par(self):
        """[n][3] routing velocity, alpha, beta of every cell's parameter set"""
        return np.array([self.catch.get(int(c), self.region_route) for c in self.cid], dtype=np.float64)

    def model(self, sb, cls=None, run=True):
        cls = cls or sb.HbvStackModel
        from shyft_b200 import synthetic
        m = cls(self.geo, catchment_parameter(self.region_route))
        for c, v in self.catch.items():
            m.set_catchment_parameter(c, catchment_parameter(v))
        if run:
            m.run_interpolation(sb.InterpolationParameter(), self.ta, self.env)
            m.set_states(synthetic.default_state(2, self.n))
            m.run_cells()
        m.set_river_network(self.rivers)
        return m

    def ups(self, r):
        return [int(u) for u in sorted(self.rivers[self.rivers[:, 1] == r, 0])]


def region(name):
    return Region(*CASES[name])


def flows(m, rivers):
    return {int(r): (m.river_local_inflow_m3s(int(r)), m.river_upstream_inflow_m3s(int(r)), m.river_output_flow_m3s(int(r)))
            for r in rivers[:, 0]}


def _uhg(capi, n, alpha, beta):
    got = capi.host_eval(2, [n, alpha, beta], max(n, 1) + 1)
    return got[1:1 + int(got[0])]


def check_against_oracle(oracle, label, reg, q, got):
    for r, (local, up, out) in got.items():
        want = oracle.river_flows(reg.rivers, r, q, reg.rid, reg.geo["routing_distance"], reg.cell_par(), reg.dt * 10**6)
        for kernel, what, g, w in (("local", "local inflow", local, want[0]), ("network", "upstream inflow", up, want[1]),
                                   ("network", "output", out, want[2])):
            n_bad, worst, where = parity_report(g, w, RTOL)
            _note((kernel, label), "oracle", np.max(np.abs(g - w)) / max(np.max(np.abs(w)), 1e-300))
            assert n_bad == 0, f"{label} river {r} {what} vs oracle: {n_bad} values outside rtol {RTOL:g}, worst {worst:.3e} at step {where}: " \
                               f"got {g[where]!r} want {w[where]!r}.  So far: {_worst_table()}"


def check_against_exact(label, reg, q, got):
    from shyft_b200 import capi
    steps = R.sample_steps(reg.T)
    par = reg.cell_par()
    n_steps = [int(capi.host_eval(3, [d, p[0], reg.dt * 10**6], 1)[0]) for d, p in zip(reg.geo["routing_distance"], par)]
    w_cell = [_uhg(capi, n, p[1], p[2]) for n, p in zip(n_steps, par)]
    for r, down, dist, vel, alpha, beta in reg.rivers:
        r = int(r)
        local, up, out = got[r]
        cells = np.flatnonzero(reg.rid == r)
        lx, lmag = R.local_exact(q, cells, w_cell, steps)
        n_chunks = max(1, math.ceil(len(cells) / 128))
        K = max((len(w_cell[c]) for c in cells), default=1) + math.ceil(min(len(cells), 128) / 32) + 5 + n_chunks
        err = np.abs(local[steps] - lx)
        _note(("local", label), "exact", np.max(err / np.maximum(R.U * lmag, 1e-300)))
        assert np.all(err <= K * R.U * lmag), f"{label} river {r} local inflow vs exact: beyond {K} ulps.  So far: {_worst_table()}"
        ups = reg.ups(r)
        w = _uhg(capi, int(capi.host_eval(3, [dist, vel, reg.dt * 10**6], 1)[0]), alpha, beta)
        ux, umag, ox, omag = R.river_exact(local, [got[u][2] for u in ups], w, steps)
        K = len(w) + len(ups) + 1
        for what, g, x, mag in (("upstream inflow", up[steps], ux, umag), ("output", out[steps], ox, omag)):
            err = np.abs(g - x)
            _note(("network", label), "exact", np.max(err / np.maximum(R.U * mag, 1e-300)))
            assert np.all(err <= K * R.U * mag), f"{label} river {r} {what} vs exact: beyond {K} ulps.  So far: {_worst_table()}"


def check(sb, oracle, label, reg, m=None):
    m = m or reg.model(sb)
    q = m.response("avg_discharge")
    got = flows(m, reg.rivers)
    check_against_oracle(oracle, label, reg, q, got)
    check_against_exact(label, reg, q, got)
    return m, got


# ---- the cases ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_routing_case(sb, oracle, name):
    reg = region(name)
    m, got = check(sb, oracle, name, reg)
    for r, (local, up, out) in got.items():
        assert np.all(np.isfinite(out)), r
        if not reg.ups(r):
            assert np.all(up == 0.0), r
    assert any(got[r][2].max() > 0 for r in got)


def test_the_cases_cover_the_edges():
    per_river, cell_taps, river_taps, Ts, dts, widest_fan, mixed_warp = set(), set(), set(), set(), set(), 0, False
    for name, (T, dt, rivers, groups, catch) in CASES.items():
        reg = region(name)
        Ts.add(T)
        dts.add(dt)
        river_taps |= {r[2] for r in rivers}
        cell_taps |= set(reg.taps[reg.rid > 0].tolist())
        for r in reg.rivers[:, 0]:
            cells = np.flatnonzero(reg.rid == r)
            per_river.add(len(cells))
            widest_fan = max(widest_fan, len(reg.ups(r)))
            for w0 in range(0, len(cells), 32):
                warp = cells[w0:w0 + 32]
                pars = {tuple(p) for p in reg.cell_par()[warp]}
                if len(pars) > 1 and len(set(reg.taps[warp])) > 1 and any(p[2] < 0 for p in pars):
                    mixed_warp = True
    assert {1, 31, 128, 129, 300, 0} <= per_river
    assert {1, 2, 24, 64, 65, 137} <= cell_taps
    assert {1, 3, 64, 65, 200, 1000} <= river_taps and 1000 > CASES["tree5_15min"][0]
    assert {1, 63, 64, 65, 999} <= Ts and dts == {900, 3600, 10800}
    assert widest_fan >= 3 and mixed_warp
    ids = CASES["tree5_15min"][2]
    assert [r[0] for r in ids] == sorted((r[0] for r in ids), reverse=True)
    assert [r[0] for r in CASES["fan3_mixed"][2]] != sorted(r[0] for r in CASES["fan3_mixed"][2])


# ---- windows ----------------------------------------------------------------------------------------------------------------------------
def windowed_region(H):
    """three rivers; the longest cell unit hydrograph has H + 1 taps, so the windowed run carries H rows of history"""
    return Region(400, 3600, [(1, 3, 3, 1.0, 7.0, 0.0), (2, 3, 65, 1.0, 3.0, 0.0), (3, 0, 24, 1.0, 7.0, 0.0)],
                  [(1, 129, (11, 12, 13), (2, H + 1, 24)), (2, 31, 1, 24), (3, 1, 1, 1), (0, 5, 1, 2)], MIXED, seed=H)


@pytest.mark.parametrize("H", [23, 136])
def test_windowed_routing_is_bit_identical_to_resident(sb, H):
    """for a given (river, step) the local-inflow kernel adds the same products in the same order whatever the time tile or window, and
    the history rows carried from window to window hold the discharge of the steps before the window: local inflow and output must not
    change a bit, for windows shorter than, as long as and longer than the history"""
    from shyft_b200 import synthetic
    reg = windowed_region(H)
    assert reg.taps.max() == H + 1
    a = reg.model(sb, sb.HbvStackOptModel)
    want = flows(a, reg.rivers)
    for window in (1, H - 1, H, H + 1, 64, 333):
        b = reg.model(sb, sb.HbvStackOptModel, run=False)
        b.initialize_cell_environment(reg.ta)
        b.set_states(synthetic.default_state(2, reg.n))
        b.run_windowed(sb.InterpolationParameter(), env=reg.env, window_steps=window)
        assert np.array_equal(a.catchment_discharges(), b.catchment_discharges()), window
        for r in reg.rivers[:, 0]:
            r = int(r)
            assert np.array_equal(b.river_local_inflow_m3s(r), want[r][0]), (window, r, "local inflow")
            assert np.array_equal(b.river_output_flow_m3s(r), want[r][2]), (window, r, "output")


# ---- parameter changes --------------------------------------------------------------------------------------------------------------
def test_a_routing_parameter_change_reroutes_the_rivers(sb, oracle):
    """river flows follow the routing velocity / alpha / beta in force when they are asked for, as the reference evaluates them lazily:
    after set_catchment_parameter or set_region_parameter the next query equals a fresh model with those parameters and the oracle.  After
    a windowed run the cell discharge of earlier windows is gone, so the query after such a change is refused"""
    reg = region("t63")
    m = reg.model(sb)
    before = flows(m, reg.rivers)
    changed = dict(reg.catch)
    changed[11] = (0.6, 0.6, -0.02)                    # 65 taps -> 108
    m.set_catchment_parameter(11, catchment_parameter(changed[11]))
    reg.catch = changed
    got = flows(m, reg.rivers)
    fresh = flows(reg.model(sb), reg.rivers)
    for r in got:
        for k in range(3):
            assert np.array_equal(got[r][k], fresh[r][k]), (r, k)
    assert not np.array_equal(got[1][0], before[1][0])
    check(sb, oracle, "t63 catchment change", reg, m)
    reg.region_route = (0.5, 1.5, 0.0)                 # the cell of catchment 1 (no override): 1 tap -> 2
    m.set_region_parameter(catchment_parameter(reg.region_route))
    got = flows(m, reg.rivers)
    fresh = flows(reg.model(sb), reg.rivers)
    for r in got:
        for k in range(3):
            assert np.array_equal(got[r][k], fresh[r][k]), (r, k)
    assert not np.array_equal(got[2][0], before[2][0])
    check(sb, oracle, "t63 region change", reg, m)
    # windowed
    from shyft_b200 import synthetic
    w = reg.model(sb, sb.HbvStackOptModel, run=False)
    w.initialize_cell_environment(reg.ta)
    w.set_states(synthetic.default_state(2, reg.n))
    w.run_windowed(sb.InterpolationParameter(), env=reg.env, window_steps=20)
    assert np.array_equal(w.river_output_flow_m3s(2), got[2][2])
    w.set_catchment_parameter(12, catchment_parameter((1.0, 7.0, 0.0)))
    with pytest.raises(RuntimeError, match="river flows need avg_discharge over the whole time axis"):
        w.river_output_flow_m3s(2)
    w.set_region_parameter(catchment_parameter(reg.region_route))
    with pytest.raises(RuntimeError, match="river flows need avg_discharge over the whole time axis"):
        w.river_local_inflow_m3s(1)


# ---- guards ---------------------------------------------------------------------------------------------------------------------------
def test_unit_hydrograph_length_guards(sb, oracle):
    """the local-inflow tile holds 64 + L_cell - 1 rows of 128 cells in at most 200 KB: a cell UHG of 137 taps runs, 138 is refused and
    the model stays usable.  A river UHG never goes through that tile: 1000 taps run with cells of at most 24 taps"""
    reg = Region(200, 3600, [(1, 2, 3, 1.0, 7.0, 0.0), (2, 0, 1, 1.0, 7.0, 0.0)], [(1, 33, 1, 137), (2, 31, 1, 24)], {})
    m, _ = check(sb, oracle, "cell137", reg)
    assert reg.taps.max() == 137
    reg.region_route = (137 / 138, 7.0, 0.0)           # the 137-tap cells now take 138 steps
    m.set_region_parameter(catchment_parameter(reg.region_route))
    with pytest.raises(RuntimeError, match="unit hydrograph too long"):
        m.river_output_flow_m3s(2)
    reg.region_route = tuple(HBV_DEFAULT[ROUTE])
    m.set_region_parameter(catchment_parameter(reg.region_route))
    check(sb, oracle, "cell137", reg, m)
    reg = Region(1100, 3600, [(1, 2, 1000, 1.0, 7.0, 0.0), (2, 0, 1000, 1.0, 3.0, 0.1)], [(1, 31, 1, 24), (2, 129, 1, 2)], {})
    check(sb, oracle, "river1000", reg)


# ---- red zones ---------------------------------------------------------------------------------------------------------------------
def red_zone_workload():
    """the smallest cases, a windowed run whose windows are shorter than the history (d_qhist, and d_rlocal rows written at g0 + t0), and
    the 137-tap cell tile"""
    import shyft_b200 as sb
    from shyft_b200 import synthetic
    for name in ("t1_3h", "t63", "t64"):
        reg = region(name)
        m = reg.model(sb)
        assert all(np.isfinite(v[2]).all() for v in flows(m, reg.rivers).values())
    reg = windowed_region(23)
    for window in (7, 23, 64):
        b = reg.model(sb, sb.HbvStackOptModel, run=False)
        b.initialize_cell_environment(reg.ta)
        b.set_states(synthetic.default_state(2, reg.n))
        b.run_windowed(sb.InterpolationParameter(), env=reg.env, window_steps=window)
        assert np.isfinite(b.river_output_flow_m3s(3)).all()
    reg = Region(70, 3600, [(1, 0, 1000, 1.0, 7.0, 0.0)], [(1, 3, 1, 137)], {})
    assert np.isfinite(flows(reg.model(sb), reg.rivers)[1][2]).all()
    print("routing paths ok")


def test_red_zones_stay_intact():
    env = dict(os.environ, SB2_GUARD="1")
    tests = os.path.join(ROOT, "tests")
    prog = f"import sys; sys.path[:0] = [{ROOT!r}, {tests!r}]; import test_gpu_routing_paths as t; t.red_zone_workload(); " \
           "from shyft_b200 import capi; v, msg = capi.check_guards(); print('guards', v, msg); sys.exit(1 if v else 0)"
    r = subprocess.run([sys.executable, "-c", prog], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "routing paths ok" in r.stdout and "guards 0" in r.stdout
