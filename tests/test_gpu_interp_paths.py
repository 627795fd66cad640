"""Every kernel run_interpolation can dispatch to, against the CPU oracle and against the exact references of interp_reference.py.

run_idw (shyft_b200/csrc/sb2_capi.cu) picks one of ten apply kernels by station count, finiteness, gradient_by_equation and, for
33-64 stations, the widest station union of a 16-cell tile (kc_max k-steps); run_btk picks one of five by the valid-station count of
each segment.  idw_kernel / btk_kernel below mirror both choices; test_the_mirror_names_the_kernels_launched checks the mirror against
the kernel names a profiler sees, and test_the_cases_cover_every_dispatch_row checks that the cases below reach every row.

IDW cases (use_idw_for_temperature = 1; max_members per variable T/P/R/W/H; "-" = 20/20/10/10/10):

    case              cells  steps    S  max_members        dispatch                          edges
    s2                    7      9    2  -                  dmma KS=4  NT=4, TMA              partial 8-cell group, 8-step row group
    s3                    1      1    3  -                  dmma KS=4  NT=4, plain            one cell, one step
    s16_flat            129     33   16  3/20/10/10/10      dmma KS=4  NT=4, TMA              flat cluster: both gradient regimes
    s17_unreached        33     65   17  -                  dmma KS=8  NT=4, plain            wind max_distance 700 m: cells without station
    s31                   9      7   31  -                  dmma KS=8  NT=4, plain            partial warp tile
    s32_long           1030    530   32  -                  dmma KS=8  NT=4, TMA              9 staging buffers, pair stores
    s33                  31      9   33  -                  compact kc<=10, plain
    s63                 129     65   63  31/20/10/10/3      compact kc>12 (T, P), kc<=10 (R, W), kc<=6 (H)
    s64_kc             1030     33   64  3/13/11/7/17       compact kc<=4 / <=10 / <=8 / <=6 / <=12, TMA
    s65                   7     33   65  -                  dmma KS=24 NT=1, plain
    s95_unreached        33      7   95  -                  dmma KS=24 NT=1, plain            wind max_distance 300 m
    s96_long            129    530   96  -                  dmma KS=24 NT=1, TMA              17 staging buffers of 32 steps
    s97                  33     65   97  -                  idw_apply_kernel                  S > 96
    s130                 31      9  130  -                  idw_apply_kernel                  S > 96
    s33_nan             129     33   33  -                  idw_apply_kernel                  5 % NaN station values
    s25_by_equation       9     65   25  6/20/10/10/10      idw_apply_kernel (T), dmma KS=8   gradient_by_equation
    (test_idw_shared_memory_guard: S = 130 at the largest max_members the 200 KB tile guard admits, and one more)

BTK cases (segments: steps x stations dropped; the valid count of each segment picks the kernel):

    case              cells  steps    S  segments                                  dispatch
    nv2                   7      9    2  9 x {}                                    dmma KS=4
    nv3                   1      7    3  7 x {}                                    dmma KS=4, odd rows (plain staging)
    nv16               1030     65   16  65 x {}                                   dmma KS=4
    nv17_long            33    530   17  530 x {}                                  dmma KS=8, 9 staging buffers
    nv32                  9     33   32  33 x {}                                   dmma KS=8
    nv33                129      9   33  9 x {}                                    dmma KS=16
    nv64                 31     65   64  65 x {}                                   dmma KS=16
    nv65               1030      7   65  7 x {}                                    dmma KS=24
    nv96_long             7    520   96  520 x {}                                  dmma KS=24, 17 staging buffers
    nv97                 33     33   97  33 x {}                                   btk_apply_kernel
    nv130               129     65  130  65 x {}                                   btk_apply_kernel
    drop17               31     56   17  9, 1 x {4}, 7, 8 x {4}, 31               KS=8 -> KS=4 -> KS=8 -> KS=4 -> KS=8
    drop33              129    106   33  33, 64 x {7}, 9                           KS=16 -> KS=8 -> KS=16
    drop65                9    136   65  65, 63 x {30}, 8                          KS=24 -> KS=16 -> KS=24
    drop97               33    103   97  7, 65 x {50}, 31                          btk_apply -> KS=24 -> btk_apply
    evict                33     40   12  2, 3 x {0}, 3 x {1} .. 3 x {9}, 3 x {0}, 3 x {5}, 2
                                         eleven valid sets through the 8-entry operator cache; {0} is evicted, then rebuilt

Every case is checked (a) against the oracle over all cells and steps: rtol 1e-13 for the dense IDW kernels, 1e-12 for the
per-neighbour kernel, BTK_RTOL for kriging; (b) against the exact reference on the sample of interp_reference.sample_cells /
sample_steps, NaN pattern included: IDW within 64 ulps of the magnitude sum_s |W_cs v_ts|, kriging within the larger of 16 times the
oracle's own error on the sample and 1e-12 max|T|.  The worst errors met per kernel are printed at the end of the module and are part of
every failure message.
"""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import interp_reference as R
from e2e_cases import run_device_windows
from fixtures import FORCING, geo_matrix
from parity import parity_report

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOUR_US = 3600 * 10**6
DEFAULT_MM = dict(temperature=20, precipitation=20, radiation=10, wind_speed=10, rel_hum=10)
IDW_DENSE_RTOL, IDW_SPARSE_RTOL = 1e-13, 1e-12
# kriging was held to 1e-9; on a B200 (1000 W power limit) the kernels differ from the oracle by at most 4.5e-15 relative on values
# above 1 % of max|T| (2.3e-16 of max|T| below that, inside the 1e-13 floor of parity_report): the host builds the same S x S
# operators as the oracle
BTK_RTOL = 1e-12


# ---- the dispatch, mirrored ------------------------------------------------------------------------------------------------------
DENSE_TILE_COMPACT, DENSE_TILE_BTK = 32, 0   # steps staged per buffer: SB2_DENSE_TILE_COMPACT in sb2_capi.cu; kriging 0 = dense_tile_steps' default


def _dmma(ks, nt, mode, compact, krow, ts):
    return f"dense_apply_dmma_kernel<{ks}, {nt}, {mode}, {'true' if compact else 'false'}, {krow}, {ts}>"


def idw_kernel(n_src, all_finite, by_equation, kc_max):
    """The apply kernel run_idw launches for one variable: the dense condition of sb2_capi.cu:778 and the SB2_DENSE chain of
    sb2_capi.cu:816-825.  by_equation is the temperature's gradient_by_equation; kc_max matters for 33-64 stations only."""
    if not all_finite or by_equation or n_src > 96:
        return "idw_apply_kernel"
    if n_src <= 16:
        return _dmma(4, 4, 0, True, 4, 0)
    if n_src <= 32:
        return _dmma(8, 4, 0, True, 8, 0)
    if n_src <= 64:
        for ks in (4, 6, 8, 10, 12):
            if kc_max <= ks:
                return _dmma(ks, 2, 0, True, 16, DENSE_TILE_COMPACT)
        return _dmma(16, 2, 0, True, 16, 0)
    return _dmma(24, 1, 0, True, 24, 0)


def btk_kernel(n_valid):
    """The apply kernel run_btk launches for a segment with n_valid stations: sb2_capi.cu:940-949."""
    if n_valid <= 16:
        return _dmma(4, 4, 1, False, 4, 0)
    if n_valid <= 32:
        return _dmma(8, 4, 1, False, 8, 0)
    if n_valid <= 64:
        return _dmma(16, 2, 1, False, 16, DENSE_TILE_BTK)
    if n_valid <= 96:
        return _dmma(24, 1, 1, False, 24, 0)
    return "btk_apply_kernel"


IDW_ROWS = {idw_kernel(s, True, False, 0) for s in (16, 32, 96)} | {idw_kernel(64, True, False, kc) for kc in (4, 6, 8, 10, 12, 16)} \
    | {"idw_apply_kernel"}
BTK_ROWS = {btk_kernel(nv) for nv in (16, 32, 64, 96, 97)}


def kc_max(src_xyz, dst_xyz, par, oracle):
    """widest station union of a 16-cell tile in k-steps of four (idw_union_plan_kernel): the stations with a non-zero dense weight for
    any cell of the tile; a cell without a station in reach has a NaN weight on station 0, which counts"""
    idx, w, cnt = oracle.idw_neighbours(src_xyz, dst_xyz, par)
    widest = 0
    for t0 in range(0, dst_xyz.shape[0], 16):
        union = set()
        for c in range(t0, min(t0 + 16, dst_xyz.shape[0])):
            union.update(idx[c, :cnt[c]].tolist() if cnt[c] else [0])
        widest = max(widest, math.ceil(len(union) / 4))
    return widest


# ---- cases -------------------------------------------------------------------------------------------------------------------------
IDW_CASES = {   # name: (cells, steps, S, config_index, options)
    "s2": (7, 9, 2, 31, {}),
    "s3": (1, 1, 3, 32, {}),
    "s16_flat": (129, 33, 16, 33, dict(mm=dict(temperature=3), flat=True)),
    "s17_unreached": (33, 65, 17, 34, dict(wind_max_distance=700.0)),
    "s31": (9, 7, 31, 35, {}),
    "s32_long": (1030, 530, 32, 36, {}),
    "s33": (31, 9, 33, 21, {}),
    "s63": (129, 65, 63, 22, dict(mm=dict(temperature=31, rel_hum=3))),
    "s64_kc": (1030, 33, 64, 23, dict(mm=dict(temperature=3, precipitation=13, radiation=11, wind_speed=7, rel_hum=17))),
    "s65": (7, 33, 65, 37, {}),
    "s95_unreached": (33, 7, 95, 38, dict(wind_max_distance=300.0)),
    "s96_long": (129, 530, 96, 39, {}),
    "s97": (33, 65, 97, 41, {}),
    "s130": (31, 9, 130, 42, {}),
    "s33_nan": (129, 33, 33, 43, dict(nan_fraction=0.05)),
    "s25_by_equation": (9, 65, 25, 44, dict(mm=dict(temperature=6), by_equation=True)),
}
EVICT = [(2, [])] + [(3, [k]) for k in range(10)] + [(3, [0]), (3, [5]), (2, [])]
BTK_CASES = {   # name: (cells, S, config_index, segments [(steps, dropped stations)])
    "nv2": (7, 2, 51, [(9, [])]),
    "nv3": (1, 3, 52, [(7, [])]),
    "nv16": (1030, 16, 53, [(65, [])]),
    "nv17_long": (33, 17, 54, [(530, [])]),
    "nv32": (9, 32, 55, [(33, [])]),
    "nv33": (129, 33, 56, [(9, [])]),
    "nv64": (31, 64, 57, [(65, [])]),
    "nv65": (1030, 65, 58, [(7, [])]),
    "nv96_long": (7, 96, 59, [(520, [])]),
    "nv97": (33, 97, 60, [(33, [])]),
    "nv130": (129, 130, 61, [(65, [])]),
    "drop17": (31, 17, 62, [(9, []), (1, [4]), (7, []), (8, [4]), (31, [])]),
    "drop33": (129, 33, 63, [(33, []), (64, [7]), (9, [])]),
    "drop65": (9, 65, 64, [(65, []), (63, [30]), (8, [])]),
    "drop97": (33, 97, 65, [(7, []), (65, [50]), (31, [])]),
    "evict": (33, 12, 66, EVICT),
}

WORST = {}   # kernel -> {"oracle": worst relative error, "exact": worst error in the unit of its bound}


def _note(kernel, what, value):
    d = WORST.setdefault(kernel, {})
    d[what] = max(d.get(what, 0.0), float(value))


def _oracle_errors(kernels, got, want):
    """record max|got - want| / max|want| and the worst relative error among values above 1 % of max|want|"""
    ok = ~np.isnan(want) & ~np.isnan(got)
    scale = np.max(np.abs(want[ok]), initial=0.0)
    if scale == 0:
        return
    d = np.abs(got[ok] - want[ok])
    big = np.abs(want[ok]) >= 0.01 * scale
    for k in kernels:
        _note(k, "oracle", np.max(d) / scale)
        _note(k, "oracle_rel", np.max(d[big] / np.abs(want[ok][big]), initial=0.0))


def _worst_table():
    return "; ".join(f"{k}: oracle {v.get('oracle', 0):.2e} / {v.get('oracle_rel', 0):.2e}, exact {v.get('exact', 0):.2e}"
                     for k, v in sorted(WORST.items()))


@pytest.fixture(scope="module", autouse=True)
def _report_worst_errors():
    yield
    print("\nworst errors per kernel (oracle: of max|want| / relative above 1 % of it; exact: IDW in ulps of the magnitude, BTK of max|T|)")
    for k, v in sorted(WORST.items()):
        print(f"  {k:48s} oracle {v.get('oracle', 0):.3e} / {v.get('oracle_rel', 0):.3e}   exact {v.get('exact', 0):.3e}")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


def idw_setup(sb, oracle, name, shape=None):
    """-> (geo, ta, env, device InterpolationParameter, oracle parameters per variable)"""
    from shyft_b200 import synthetic
    n, T, S, cfg, o = IDW_CASES[name]
    n, T = shape or (n, T)
    geo, ta, env = synthetic.make_region(n, T, S, config_index=cfg, nan_fraction=o.get("nan_fraction", 0.0))
    if o.get("flat"):   # half the stations within 4 m of each other: cells that only see them take the default gradient
        xyz = env.temperature[0].copy()
        xyz[: S // 2, 2] = 500.0 + np.arange(S // 2) * 0.5
        env.temperature = (xyz, env.temperature[1])
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    pars = {}
    for var in FORCING:
        mm = o.get("mm", {}).get(var, DEFAULT_MM[var])
        dev = getattr(ip, "temperature_idw" if var == "temperature" else var)
        dev.max_members = mm
        kw = dict(max_members=mm)
        if var == "wind_speed" and "wind_max_distance" in o:
            dev.max_distance = kw["max_distance"] = o["wind_max_distance"]
        if var == "temperature" and o.get("by_equation"):
            dev.gradient_by_equation = 1
            kw["gradient_by_equation"] = True
        pars[var] = oracle.idw_par(**kw)
    return geo, ta, env, ip, pars


def idw_kernels_of(oracle, name, geo, env, pars):
    gm = geo_matrix(geo)
    S = IDW_CASES[name][2]
    out = {}
    for var in FORCING:
        xyz, vals = getattr(env, var)
        kc = kc_max(xyz, gm[:, :3], pars[var], oracle) if 32 < S <= 64 else 0
        out[var] = idw_kernel(S, bool(np.all(np.isfinite(vals))), var == "temperature" and bool(pars[var][5]), kc)
    return out


def btk_setup(sb, name, n=None, segments=None):
    from shyft_b200 import synthetic
    n0, S, cfg, segs = BTK_CASES[name]
    n, segs = n or n0, segments or segs
    T = sum(length for length, _ in segs)
    geo, ta, env = synthetic.make_region(n, T, S, config_index=cfg)
    xyz, vals = env.temperature
    vals = vals.copy()
    t = 0
    for length, dropped in segs:
        vals[t:t + length, dropped] = np.nan
        t += length
    env.temperature = (xyz, vals)
    return geo, ta, env, sb.InterpolationParameter()


def btk_kernels_of(vals):
    return [btk_kernel(int(np.isfinite(vals[a]).sum())) for a, b in R.segments(vals)]


def _interpolate(sb, geo, ta, env, ip):
    m = sb.PTGSKOptModel(geo)
    assert m.run_interpolation(ip, ta, env, best_effort=False)
    return m


def check_idw(oracle, name, kernel, got, var, env, geo, par):
    """(a) oracle over everything, (b) exact reference on the sample"""
    gm = geo_matrix(geo)
    xyz, vals = getattr(env, var)
    vals = oracle.average_accessor_same_axis(vals, HOUR_US)
    want = oracle.idw_run(var, xyz, vals, gm[:, :3], par, dst_slope=gm[:, 5], ncore=8)
    rtol = IDW_SPARSE_RTOL if kernel == "idw_apply_kernel" else IDW_DENSE_RTOL
    n_bad, worst, where = parity_report(got, want, rtol)
    _oracle_errors([kernel], got, want)
    assert n_bad == 0, f"{name} {var} ({kernel}) vs oracle: {n_bad} values outside rtol {rtol:g}, worst {worst:.3e} at {where}: " \
                       f"got {got[where]!r} want {want[where]!r}.  So far: {_worst_table()}"
    cells, steps = R.sample_cells(got.shape[1]), R.sample_steps(got.shape[0])
    exact, mag = R.idw_exact(oracle, var, xyz, vals, gm[:, :3], par, cells, steps, dst_slope=gm[:, 5])
    g = got[np.ix_(steps, cells)]
    assert np.array_equal(np.isnan(g), np.isnan(exact)), f"{name} {var}: NaN pattern differs from the exact reference"
    ok = ~np.isnan(exact)
    err, bound = np.abs(g - exact)[ok], 64 * R.U * mag[ok]
    if var == "temperature" and par[5]:
        # the 3x3 plane fit amplifies round-off by its condition number, on the device as in the oracle: allow 16 times the oracle's
        # own error on the same sample on top of the summation bound
        o = want[np.ix_(steps, cells)][ok]
        bound = bound + 16 * np.max(np.abs(o - exact[ok]))
    ratio = np.max(err / np.maximum(R.U * mag[ok], 1e-300), initial=0.0)
    _note(kernel, "exact", ratio)
    assert np.all(err <= bound), f"{name} {var} ({kernel}) vs exact: worst {ratio:.1f} ulps of the magnitude.  So far: {_worst_table()}"


def check_btk(oracle, name, got, geo, ta, env):
    gm = geo_matrix(geo)
    xyz, vals = env.temperature
    vals = oracle.average_accessor_same_axis(vals, HOUR_US)
    want = oracle.btk_run(xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US)
    kernels = btk_kernels_of(vals)
    n_bad, worst, where = parity_report(got, want, BTK_RTOL)
    _oracle_errors(kernels, got, want)
    assert n_bad == 0, f"{name} ({kernels}) vs oracle: {n_bad} values outside rtol {BTK_RTOL:g}, worst {worst:.3e} at {where}: " \
                       f"got {got[where]!r} want {want[where]!r}.  So far: {_worst_table()}"
    cells, steps = R.sample_cells(got.shape[1]), R.btk_sample_steps(vals)
    exact = R.btk_exact(oracle, xyz, vals, gm[:, :3], ta.start * 10**6, HOUR_US, cells, steps)
    g, o = got[np.ix_(steps, cells)], want[np.ix_(steps, cells)]
    assert np.array_equal(np.isnan(g), np.isnan(exact))
    scale = np.max(np.abs(exact))
    err_dev, err_oracle = np.max(np.abs(g - exact)), np.max(np.abs(o - exact))
    for k in kernels:
        _note(k, "exact", err_dev / scale)
    bound = max(16 * err_oracle, 1e-12 * scale)
    assert err_dev <= bound, f"{name} ({kernels}) vs exact: {err_dev / scale:.3e} of max|T| (oracle {err_oracle / scale:.3e}).  " \
                             f"So far: {_worst_table()}"


# ---- IDW -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(IDW_CASES))
def test_idw_case(sb, oracle, name):
    geo, ta, env, ip, pars = idw_setup(sb, oracle, name)
    kernels = idw_kernels_of(oracle, name, geo, env, pars)
    m = _interpolate(sb, geo, ta, env, ip)
    for var in FORCING:
        check_idw(oracle, name, kernels[var], m.cell_forcing(var), var, env, geo, pars[var])
    o = IDW_CASES[name][4]
    if "wind_max_distance" in o:
        w = m.cell_forcing("wind_speed")
        assert np.isnan(w).any() and not np.isnan(w).all()
    if o.get("flat"):
        gm = geo_matrix(geo)
        xyz = env.temperature[0]
        idx, _, cnt = oracle.idw_neighbours(xyz, gm[:, :3], pars["temperature"])
        span = np.array([np.ptp(xyz[idx[c, :cnt[c]], 2]) for c in range(len(geo))])
        assert (span <= 50).any() and (span > 50).any()


def test_idw_shared_memory_guard(sb, oracle):
    """S = 130 runs per neighbour; the largest max_members whose tiles fit the 200 KB guard of run_idw works, one more is refused with
    the guard's message, and the model stays usable (no CUDA error behind it)"""
    n, T, S = 31, 9, 130
    tile = max(1, min(64, 4096 // S))                      # idw_tile_steps
    largest = (200 * 1024 - tile * S * 8) // (128 * 20)    # max_k * IDW_BLOCK * (2 doubles + 1 int) on top of the station tile
    assert largest < S
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, S, config_index=42)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    m = sb.PTGSKOptModel(geo)
    ip.precipitation.max_members = largest + 1
    with pytest.raises(RuntimeError, match="too many sources / members for the shared-memory tiles"):
        m.run_interpolation(ip, ta, env, best_effort=False)
    ip.precipitation.max_members = largest
    assert m.run_interpolation(ip, ta, env, best_effort=False)
    check_idw(oracle, "guard", "idw_apply_kernel", m.cell_forcing("precipitation"), "precipitation", env, geo,
              oracle.idw_par(max_members=largest))


# ---- BTK -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(BTK_CASES))
def test_btk_case(sb, oracle, name):
    geo, ta, env, ip = btk_setup(sb, name)
    m = _interpolate(sb, geo, ta, env, ip)
    check_btk(oracle, name, m.cell_forcing("temperature"), geo, ta, env)


# ---- dispatch coverage -------------------------------------------------------------------------------------------------------------
def test_the_cases_cover_every_dispatch_row(sb, oracle):
    idw_hit, btk_hit = set(), set()
    for name in IDW_CASES:
        geo, ta, env, ip, pars = idw_setup(sb, oracle, name)
        idw_hit |= set(idw_kernels_of(oracle, name, geo, env, pars).values())
    for name in BTK_CASES:
        btk_hit |= set(btk_kernels_of(btk_setup(sb, name)[2].temperature[1]))
    assert idw_hit == IDW_ROWS, f"IDW rows not covered: {sorted(IDW_ROWS - idw_hit)}"
    assert btk_hit == BTK_ROWS, f"BTK rows not covered: {sorted(BTK_ROWS - btk_hit)}"
    assert len(IDW_ROWS) == 10 and len(BTK_ROWS) == 5
    kc = {idw_kernel(64, True, False, k) for k in (4, 6, 8, 10, 12, 13)}
    assert kc <= idw_hit                                        # all six variants of the 33-64 bin
    for a, b in zip(EVICT, EVICT[1:]):
        assert a[1] != b[1]
    assert len({tuple(d) for _, d in EVICT}) > 8                # more valid sets than the operator cache holds


def _plain(kernel):
    """'void sb2::idw_apply_kernel<2>(long, ...)' -> 'idw_apply_kernel'; template arguments of the dense kernel kept, blanks dropped"""
    k = re.sub(r"\s", "", kernel.split("(")[0]).removeprefix("void").replace("sb2::", "")
    return re.sub(r"^idw_apply_kernel<\d+>$", "idw_apply_kernel", k)


def _launched_apply_kernels(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {_plain(e.name) for e in prof.events() if re.search(r"(dense_apply_dmma|idw_apply|btk_apply)_kernel", e.name)}


def test_the_mirror_names_the_kernels_launched(sb, oracle):
    """idw_kernel / btk_kernel against the kernel names the CUDA profiler records, for one small case of every row"""
    for name in ("s3", "s31", "s33", "s63", "s64_kc", "s65", "s97", "s25_by_equation"):
        n, T = IDW_CASES[name][:2]
        geo, ta, env, ip, pars = idw_setup(sb, oracle, name, shape=(n, min(T, 9)))
        want = {_plain(k) for k in idw_kernels_of(oracle, name, geo, env, pars).values()}
        got = _launched_apply_kernels(lambda: _interpolate(sb, geo, ta, env, ip))
        assert got == want, (name, sorted(got), sorted(want))
    for name in ("drop17", "drop65", "drop97"):
        geo, ta, env, ip = btk_setup(sb, name)
        S = BTK_CASES[name][1]
        gm = geo_matrix(geo)
        want = set(btk_kernels_of(env.temperature[1]))
        for var in FORCING[1:]:     # the other four variables: IDW with the default parameters
            par = oracle.idw_par(max_members=DEFAULT_MM[var])
            want.add(idw_kernel(S, True, False, kc_max(getattr(env, var)[0], gm[:, :3], par, oracle) if 32 < S <= 64 else 0))
        got = _launched_apply_kernels(lambda: _interpolate(sb, geo, ta, env, ip))
        assert got == {_plain(k) for k in want}, (name, sorted(got), sorted(want))


# ---- windows and the catchment filter -------------------------------------------------------------------------------------------------
WINDOWED = [("idw", "s33", 129, 130), ("btk", "drop33", None, None), ("btk", "nv130", 129, 130)]


@pytest.mark.parametrize("kind,name,n,T", WINDOWED, ids=[w[1] for w in WINDOWED])
def test_windowed_forcing_is_bit_identical_to_one_shot(sb, oracle, kind, name, n, T):
    """A step's DMMA k-order does not depend on where the step sits in a staging buffer, and the prior gradient is indexed by absolute
    step, so cutting the axis into windows (each window one launch per segment) must not change a bit"""
    from shyft_b200 import synthetic
    if kind == "idw":
        geo, ta, env, ip, _ = idw_setup(sb, oracle, name, shape=(n, T))
    else:
        segs = None if T is None else [(T, [])]
        geo, ta, env, ip = btk_setup(sb, name, n=n, segments=segs)
    T = ta.n
    one = _interpolate(sb, geo, ta, env, ip)
    ref = {k: one.cell_forcing(k) for k in FORCING}
    for window in (1, 7, 33, 65, 777):
        m = sb.PTGSKOptModel(geo)
        m.initialize_cell_environment(ta)
        m._set_sources(env)
        m.set_states(synthetic.default_state(0, len(geo)))
        got = {k: np.full_like(ref[k], -1.0) for k in FORCING}

        def keep(w0, _resp, forcing):
            for k in FORCING:
                got[k][w0:w0 + forcing[k].shape[0]] = forcing[k]
        run_device_windows(m, ip, T, window, (), (), keep)
        for k in FORCING:
            same = (got[k] == ref[k]) | (np.isnan(got[k]) & np.isnan(ref[k]))
            assert same.all(), f"{name} window {window} {k}: {np.count_nonzero(~same)} values differ, first at {np.argwhere(~same)[0]}"


@pytest.mark.parametrize("kind,name", [("idw", "s17_unreached"), ("btk", "nv16"), ("idw", "s97")])
def test_catchment_filter_leaves_half_pairs_alone(sb, oracle, kind, name):
    """alternating catchment ids: the filter keeps one cell of every stored pair; the inactive ones keep their NaN fill, the active ones
    equal the unfiltered run bit for bit (dense IDW, kriging DMMA and per-neighbour IDW), in one shot and window by window"""
    n, T = 33, 33
    if kind == "idw":
        geo, ta, env, ip, _ = idw_setup(sb, oracle, name, shape=(n, T))
    else:
        geo, ta, env, ip = btk_setup(sb, name, n=n, segments=[(T, [])])
    geo = geo.copy()
    geo["catchment_id"] = 1 + np.arange(n) % 2
    full = _interpolate(sb, geo, ta, env, ip)
    m = sb.PTGSKOptModel(geo)
    m.set_catchment_calculation_filter([2])
    assert m.run_interpolation(ip, ta, env, best_effort=False)
    active = np.arange(n) % 2 == 1
    for k in FORCING:
        a, b = m.cell_forcing(k), full.cell_forcing(k)
        assert np.isnan(a[:, ~active]).all(), k
        assert np.array_equal(a[:, active], b[:, active], equal_nan=True), k
    # windowed: the window buffers are reused, also those an unfiltered interpolation of the whole axis filled (window_steps == T)
    from shyft_b200 import synthetic
    for window in (T, 7):
        w = sb.PTGSKOptModel(geo)
        assert w.run_interpolation(ip, ta, env, best_effort=False)
        w.set_catchment_calculation_filter([2])
        w.set_states(synthetic.default_state(0, n))
        got = {k: np.zeros((T, n)) for k in FORCING}

        def keep(w0, _resp, forcing):
            for k in FORCING:
                got[k][w0:w0 + forcing[k].shape[0]] = forcing[k]
        run_device_windows(w, ip, T, window, (), (), keep)
        for k in FORCING:
            assert np.isnan(got[k][:, ~active]).all(), (window, k)
            assert np.array_equal(got[k][:, active], full.cell_forcing(k)[:, active], equal_nan=True), (window, k)


# ---- red zones ---------------------------------------------------------------------------------------------------------------------
def red_zone_workload():
    """the smallest odd shapes of every path: 7 cells x 9 steps, odd and even S per bin, the six compaction variants, NaN and
    gradient_by_equation per-neighbour IDW, every kriging kernel and one drop-out run across a bin"""
    import shyft_b200 as sb
    from shyft_b200 import synthetic
    n, T = 7, 9
    runs = []
    for S, mm in [(2, {}), (3, {}), (16, {}), (17, {}), (31, {}), (32, {}), (33, dict(temperature=1, precipitation=3, radiation=7, wind_speed=9)),
                  (64, dict(temperature=7, precipitation=21)), (65, {}), (95, {}), (96, {}), (97, {})]:
        geo, ta, env = synthetic.make_region(n, T, S, config_index=70 + S)
        ip = sb.InterpolationParameter(use_idw_for_temperature=1)
        for var, k in mm.items():
            getattr(ip, "temperature_idw" if var == "temperature" else var).max_members = k
        runs.append((geo, ta, env, ip))
    geo, ta, env = synthetic.make_region(n, T, 33, config_index=90, nan_fraction=0.05)
    ip = sb.InterpolationParameter(use_idw_for_temperature=1)
    ip.temperature_idw.gradient_by_equation = 1
    runs.append((geo, ta, env, ip))
    for S in (2, 3, 16, 17, 32, 33, 64, 65, 96, 97):
        geo, ta, env = synthetic.make_region(n, T, S, config_index=100 + S)
        runs.append((geo, ta, env, sb.InterpolationParameter()))
    geo, ta, env = synthetic.make_region(n, T, 97, config_index=91)
    xyz, vals = env.temperature
    vals = vals.copy()
    vals[3:6, 50] = np.nan                                     # 97 -> 96 -> 97 stations
    env.temperature = (xyz, vals)
    runs.append((geo, ta, env, sb.InterpolationParameter()))
    for geo, ta, env, ip in runs:
        m = sb.PTGSKOptModel(geo)
        m.run_interpolation(ip, ta, env, best_effort=False)
        for k in FORCING:
            assert np.isfinite(m.cell_forcing(k)).any(), k
    print("interp paths ok")


def test_red_zones_stay_intact():
    env = dict(os.environ, SB2_GUARD="1")
    tests = os.path.join(ROOT, "tests")
    prog = f"import sys; sys.path[:0] = [{ROOT!r}, {tests!r}]; import test_gpu_interp_paths as t; t.red_zone_workload(); " \
           "from shyft_b200 import capi; v, msg = capi.check_guards(); print('guards', v, msg); sys.exit(1 if v else 0)"
    r = subprocess.run([sys.executable, "-c", prog], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "interp paths ok" in r.stdout and "guards 0" in r.stdout
