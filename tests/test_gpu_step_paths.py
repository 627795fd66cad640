"""Every launch path of the five cell stacks' step kernels against the oracle, bit for bit (DESIGN.md section 2), at the edges where a
launcher goes wrong: ragged warps and time slices, the time split switched off (16 000 step groups and more), chunks of a resident
run, the parameter-table instantiations with parameter sets mixed inside a warp, the calculation filter, every collector mode, and
the pt_gs_k calibration batch at and beyond its split threshold.  Catchment sums are held to the exact sum of the device's own
per-cell series within the bound any summation order meets (tests/step_cases.py).

Each case shows which path it took: the CUDA profiler records the kernel names (the template arguments name the collector mode and
the parameter source) and grids (step groups x time slices when split, step groups when not)."""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import pytest

import step_cases as sc
from fixtures import FORCING, PTGSK_DEFAULT, geo_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H = 3600 * 10**6
DAY = 86400
WINTER = 1424476800   # 2015-02-21: snowfall and a snow pack from the first step
K_MMH_M3S = 1.0 / (3600.0 * 1000.0)

# case A: (n, T) around the 32-cell warp and the 64- and 128-step slices
RAGGED = [(1, 1), (1, 65), (31, 63), (31, 64), (33, 65), (33, 129), (100, 1), (100, 64), (100, 129), (257, 63), (257, 65), (257, 129)]
BIG_N, BIG_T = 512017, 150        # case B: 16 001 step groups, the last one 17 cells
LONG_N, LONG_T = 70, 5000         # case C: two chunks of a resident run
SLICE_ROWS = (0, 63, 64, 65)      # state-series rows around the 64-step slice

REPORT = []   # (case, what it proved)


def note(case, what):
    REPORT.append((case, what))
    print(f"[{case}] {what}")


@pytest.fixture(scope="module", autouse=True)
def _report():
    t0 = time.perf_counter()
    yield
    print("\nstep paths proved (worst catchment-sum error in units of its bound gamma(m-1) * sum|x|):")
    for case, what in REPORT:
        print(f"  {case:28s} {what}")
    print(f"module wall time {time.perf_counter() - t0:.1f} s")


@pytest.fixture(scope="module")
def sb():
    import shyft_b200
    return shyft_b200


# ---- launched kernels ------------------------------------------------------------------------------------------------------------------
STEP_RE = re.compile(r"(ptgsk_forcing_terms|ptgsk_snow|ptgsk_response|hbv_run|ptssk_run|pthpsk_run|catchment_reduce)_kernel")


def _plain(name):
    """'void sb2::ptgsk_snow_kernel<14, true>(sb2::PtgskRunArgs)' -> 'ptgsk_snow_kernel<14,true>'"""
    return re.sub(r"\s", "", name.split("(")[0]).removeprefix("void").replace("sb2::", "")


def launched(fn):
    """run fn under the CUDA profiler -> [(plain kernel name, grid [x, y, z] or None)] of every kernel, in launch order"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # the library's first kernels in a profiler window can go unrecorded: open the window with two of its own (sb2_unit_eval)
        from shyft_b200 import capi
        for _ in range(2):
            capi.unit_eval("exp", [[0.0]])
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    ks = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return [(_plain(e["name"]), e.get("args", {}).get("grid")) for e in ks]


def step_launches(kernels):
    return [(k, g) for k, g in kernels if STEP_RE.match(k) and not k.startswith("catchment_reduce")]


def assert_path(case, stack, kernels, names, n, chunks, members=1):
    """the step kernels launched are `names` once per chunk; their grids show the split (groups x slices) or not (groups)"""
    steps = step_launches(kernels)
    got = [k for k, _ in steps]
    assert got == [k for _ in chunks for k in names], (case, got, names)
    assert sum(k.startswith("catchment_reduce") for k, _ in kernels) == len(chunks), case
    split = sc.time_split(n, members)
    grids = [g for k, g in steps if not k.startswith("ptgsk_forcing_terms")]
    if all(g is not None for g in grids):
        per = len(names) - (1 if stack == "pt_gs_k" else 0)
        want = [sc.step_grid_x(stack, n, c, members) for c in chunks for _ in range(per)]
        assert [g[0] for g in grids] == want, (case, grids, want)
        assert all(g[1] == members for g in grids), case
        how = "grid"
    else:
        how = "host rule"
    note(case, f"{stack}: {' '.join(sorted(set(names)))}; {'split' if split else 'unsplit'} ({sc.step_groups(n)} groups x {members} "
               f"members, by {how}); chunks {chunks}")


# ---- models and the oracle ---------------------------------------------------------------------------------------------------------------
def region(sb, stack, n, T, cids=None, cfg=None, cells_per_catchment=None, stations=4, cls=None):
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, stations, config_index=30 + n % 7 if cfg is None else cfg,
                                         cells_per_catchment=cells_per_catchment or max(1, n // 3), start=WINTER)
    if cids is not None:
        geo["catchment_id"] = cids
    m = getattr(sb, cls or sc.MODEL[stack])(geo, sc.DEFAULT[stack])
    assert m.run_interpolation(sb.InterpolationParameter(), ta, env)
    return m, geo, ta, env


def initial_state(m, stack, n):
    """the synthetic default state with a snow pack from the first step where the state can carry one directly"""
    from shyft_b200 import synthetic
    st = synthetic.default_state(sc.STACK_ID[stack], n)
    if stack == "pt_gs_k":
        st[:, 5] = -1.0                       # acc_melt < 0: accumulation branch
        st[:, 4] = np.linspace(5.0, 80.0, n)  # sdc_melt_mean
        st[:, 1] = 2.0                        # liquid water: wet-snow paths
    elif stack in ("pt_hs_k", "hbv_stack"):
        st[:, 0] = np.linspace(5.0, 80.0, n)  # swe and sca, distributed over the five bins as run_cells would
        st[:, 1] = 0.9
        st = m.distribute_snow(st)
    return st


def forcing(m, cells=None):
    return {k: (m.cell_forcing(k) if cells is None else np.ascontiguousarray(m.cell_forcing(k)[:, cells])) for k in FORCING}


def oracle_run(oracle, stack, gm, par, f, st, ta, n_steps=0, pset=None):
    """-> (response dict, end state, state-series dict or None): the oracle's run of these cells"""
    t0, dt = ta.start * 10**6, ta.delta_t * 10**6
    kw = dict(n_steps=n_steps, pset_of_cell=pset, ncore=8)
    if stack == "pt_gs_k":
        o = oracle.ptgsk_run_cells(gm, par, f, st, t0, dt, collect_response=True, collect_state=True, **kw)
        return {k: o[k] for k in sc.responses(stack)}, o["state"], {k: o[k] for k in oracle.PTGSK_STATES}
    if stack == "pt_ss_k":
        o = oracle.ptssk_run_cells(gm, par, f, st, t0, dt, collect_state=True, **kw)
        return {k: o[k] for k in sc.responses(stack)}, o["state"], {k[6:]: v for k, v in o.items() if k.startswith("state_")}
    fn = dict(pt_hs_k=oracle.pthsk_run_cells, hbv_stack=oracle.hbv_stack_run_cells, pt_hps_k=oracle.pthpsk_run_cells)[stack]
    o = fn(gm, par, f, st, t0, dt, **kw)
    return {k: o[k] for k in sc.responses(stack)}, o["state"], None


def state_row(stack, st, gm):
    """the state collector's values of an end state (sb2_hbv.cuh / sb2_pthpsk.cuh collect_state): name -> [n]"""
    area, ssf = gm[:, 3], 1.0 - gm[:, 7] - gm[:, 8]
    if stack == "hbv_stack":
        d = dict(snow_swe=st[:, 0], snow_sca=st[:, 1], soil_moisture=st[:, 12], tank_uz=st[:, 13], tank_lz=st[:, 14])
        sp, sw = 2, 7
    elif stack == "pt_hs_k":
        d = dict(kirchner_discharge=area * st[:, 12] * K_MMH_M3S, snow_sca=st[:, 1], snow_swe=st[:, 0] * ssf)
        sp, sw = 2, 7
    else:   # pt_hps_k
        d = dict(kirchner_discharge=area * st[:, 23] * K_MMH_M3S, snow_sca=st[:, 22], snow_swe=st[:, 21] * ssf, snow_surface_heat=st[:, 20])
        d.update({f"snow_albedo_{i}": st[:, 10 + i] for i in range(5)})
        d.update({f"snow_iso_pot_energy_{i}": st[:, 15 + i] for i in range(5)})
        sp, sw = 0, 5
    d.update({f"snow_sp_{i}": st[:, sp + i] for i in range(5)})
    d.update({f"snow_sw_{i}": st[:, sw + i] for i in range(5)})
    return d


def same(got, want, what):
    """bit identity (NaN where the other has NaN); on failure the first differing (row, cell)"""
    if np.array_equal(got, want, equal_nan=True):
        return
    bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
    i = tuple(bad[0])
    raise AssertionError(f"{what}: {len(bad)} values differ, first at {i}: got {got[i]!r} want {want[i]!r}")


class Expected:
    """the oracle's view of some cells of a model: responses, end state and the state-series rows asked for"""

    def __init__(self, oracle, stack, gm, par, f, st0, ta, rows, pset=None):
        self.resp, self.state, series = oracle_run(oracle, stack, gm, par, f, st0, ta, pset=pset)
        self.rows = {}
        for r in rows:
            if series is not None:
                self.rows[r] = {k: v[r] for k, v in series.items()}
            else:   # the HBV-family oracle keeps no state series: the end state of the run cut at row r
                st = st0 if r == 0 else (self.state if r == ta.n else oracle_run(oracle, stack, gm, par, f, st0, ta, n_steps=r, pset=pset)[1])
                self.rows[r] = state_row(stack, st, gm)


def check_cells(m, stack, want, cells, what, state_series=True, resp=None):
    """responses, the state-series rows of `want` and the end state of `cells` bit-identical to `want`"""
    for name in sc.responses(stack):
        got = resp[name] if resp is not None else m.response(name)[:, cells]
        same(got, want.resp[name], f"{what} {name}")
    if state_series:
        for r, d in want.rows.items():
            for name, v in d.items():
                same(m.state_series(name, r, 1)[0, cells], v, f"{what} state series {name} row {r}")
    same(m.get_states()[cells], want.state, f"{what} end state")


def check_sums(m, what, catchments=None):
    """catchment discharges and charges within gamma(m-1) sum|x| of the exact sum of the device's per-cell series"""
    cix = m.cell_catchment_ix()
    r = max(sc.worst_catchment_sum_ratio(m.catchment_discharges(), m.response("avg_discharge"), cix, catchments),
            sc.worst_catchment_sum_ratio(m.catchment_charges(), m.response("charge_m3s"), cix, catchments))
    assert r <= 1.0, f"{what}: a catchment sum is {r:.3g} bounds from the exact sum"
    return r


def rows_of(T, extra=()):
    return sorted({r for r in SLICE_ROWS + tuple(extra) + (T,) if r <= T})


# ---- A: ragged sizes -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stack", sc.STACKS)
@pytest.mark.parametrize("n,T", RAGGED)
def test_ragged_sizes(sb, oracle, stack, n, T):
    """one cell, one step, cell counts around the warp, step counts around both slice lengths: every series, the state rows around
    the slice and the end state bit-identical to the oracle (lanes past the last cell shadow a cell and store nothing)"""
    m, geo, ta, _ = region(sb, stack, n, T)
    st0 = initial_state(m, stack, n)
    m.set_states(st0)
    m.set_state_collection(-1, True)
    kernels = launched(m.run_cells)
    assert_path(f"A {n}x{T}", stack, kernels, sc.step_kernels(stack, 15, table=False), n, sc.run_cells_chunks(T))
    gm = geo_matrix(geo)
    want = Expected(oracle, stack, gm, sc.DEFAULT[stack], forcing(m), st0, ta, rows_of(T))
    check_cells(m, stack, want, slice(None), f"{stack} {n}x{T}")
    if stack in ("pt_gs_k", "pt_ss_k"):   # the oracle's state series in full
        _, _, series = oracle_run(oracle, stack, gm, sc.DEFAULT[stack], forcing(m), st0, ta)
        for name, v in series.items():
            same(m.state_series(name), v, f"{stack} {n}x{T} state series {name}")
    note(f"A {n}x{T}", f"{stack}: catchment sums {check_sums(m, stack):.3f}")


# ---- B: the time split off in run_cells --------------------------------------------------------------------------------------------------
def big_sample(n):
    rng = np.random.default_rng(7)
    groups = rng.choice(np.arange(1, sc.step_groups(n)), 50, replace=False)
    cells = np.concatenate([np.arange(32), np.arange(n - n % 32, n), groups * 32 - 1, groups * 32, rng.choice(n, 1900, replace=False)])
    return np.unique(cells)


@pytest.mark.parametrize("stack", sc.STACKS)
def test_time_split_off_in_run_cells(sb, oracle, stack):
    """512 017 cells = 16 001 step groups: every block steps the whole chunk.  A sample of cells (the first and the ragged last warp,
    both sides of 50 group boundaries, random cells) equals the oracle and a small model of just those cells (which time-slices)."""
    n, T = BIG_N, BIG_T
    assert not sc.time_split(n) and sc.time_split(n - 17 - 32)
    m, geo, ta, _ = region(sb, stack, n, T, cfg=11, cells_per_catchment=1000, stations=16)
    cells = big_sample(n)
    assert cells.size >= 2000
    st0 = initial_state(m, stack, n)
    m.set_states(st0)
    kernels = launched(m.run_cells)
    assert_path("B unsplit run_cells", stack, kernels, sc.step_kernels(stack, 7, table=False), n, sc.run_cells_chunks(T))
    s = m.get_states()
    assert np.all(np.isfinite(s))
    got = {}
    for name in sc.responses(stack):
        full = m.response(name)
        got[name] = np.ascontiguousarray(full[:, cells])
        del full
    ratio = check_sums(m, f"{stack} unsplit")
    f = forcing(m, cells)
    del m
    gm = geo_matrix(geo[cells])
    want = Expected(oracle, stack, gm, sc.DEFAULT[stack], f, st0[cells], ta, [])
    for name in sc.responses(stack):
        same(got[name], want.resp[name], f"{stack} unsplit {name}")
    same(s[cells], want.state, f"{stack} unsplit end state")
    # the same cells as a model of their own: 64 step groups, time-sliced
    small = getattr(sb, sc.MODEL[stack])(geo[cells], sc.DEFAULT[stack])
    small.initialize_cell_environment(ta)
    for k in FORCING:
        small.set_cell_forcing(k, f[k])
    small.set_states(st0[cells])
    kernels = launched(small.run_cells)
    assert_path("B split (sample model)", stack, kernels, sc.step_kernels(stack, 7, table=False), cells.size, sc.run_cells_chunks(T))
    for name in sc.responses(stack):
        same(small.response(name), got[name], f"{stack} sample model {name}")
    same(small.get_states(), s[cells], f"{stack} sample model end state")
    note("B unsplit run_cells", f"{stack}: {cells.size} sampled cells bit-identical; catchment sums {ratio:.3f}")


# ---- C: a resident run of two chunks, and partial ranges ----------------------------------------------------------------------------------
@pytest.mark.parametrize("stack", sc.STACKS)
def test_multi_chunk_resident_run(sb, oracle, stack):
    n, T = LONG_N, LONG_T
    chunks = sc.run_cells_chunks(T)
    assert chunks == [2560, 2440]
    m, geo, ta, _ = region(sb, stack, n, T, cfg=12, cells_per_catchment=32)
    st0 = initial_state(m, stack, n)
    m.set_states(st0)
    m.set_state_collection(-1, True)
    k0 = m.kernel_launches()
    kernels = launched(m.run_cells)
    k_two = m.kernel_launches() - k0
    assert m.step_chunk_steps() == sc.RUN_CELLS_CAP
    assert_path("C two chunks", stack, kernels, sc.step_kernels(stack, 15, table=False), n, chunks)
    gm = geo_matrix(geo)
    f = forcing(m)
    cut = (37, 4133)
    want = Expected(oracle, stack, gm, sc.DEFAULT[stack], f, st0, ta, rows_of(T, (2559, 2560, 2561) + cut))
    check_cells(m, stack, want, slice(None), f"{stack} two chunks")
    one = {name: m.response(name) for name in sc.responses(stack)}
    one_st = {name: m.state_series(name) for name in sb.capi.STATE_SERIES_NAMES[sc.STACK_ID[stack]]}
    s_end = m.get_states()
    # one chunk fewer, the same series filled: the launch counter differs by one chunk's step kernels and catchment reduction
    m.revert_to_initial_state()
    k0 = m.kernel_launches()
    m.run_cells(0, 0, sc.RUN_CELLS_CAP)
    assert k_two - (m.kernel_launches() - k0) == len(sc.step_kernels(stack, 15, table=False)) + 1
    # the same axis as three run_cells ranges: each writes its end-state row (the next range would overwrite it with the same value)
    m.revert_to_initial_state()
    for first, count in ((0, 37), (37, 4096), (4133, T - 4133)):
        m.run_cells(0, first, count)
        r = first + count
        for name, v in want.rows[r].items():
            same(m.state_series(name, r, 1)[0], v, f"{stack} state series {name} at the end of range [{first}, {r})")
    for name, v in one.items():
        same(m.response(name), v, f"{stack} ranges vs one shot {name}")
    for name, v in one_st.items():
        same(m.state_series(name), v, f"{stack} ranges vs one shot state series {name}")
    same(m.get_states(), s_end, f"{stack} ranges vs one shot end state")
    note("C two chunks", f"{stack}: rows 2559-2561 and range ends 37 / 4133 / 5000 bit-identical; catchment sums {check_sums(m, stack):.3f}")


# ---- D: the parameter-table kernels, parameter sets mixed inside a warp ---------------------------------------------------------------------
def interleaved(n):
    return 1 + np.arange(n) % 3   # catchments 1 / 2 / 3 lane by lane


@pytest.mark.parametrize("stack", sc.STACKS)
def test_parameter_table_kernels(sb, oracle, stack):
    n, T = 96, 200
    m, geo, ta, _ = region(sb, stack, n, T, cids=interleaved(n), cfg=13)
    st0 = initial_state(m, stack, n)
    m.set_states(st0)
    m.set_state_collection(-1, True)
    over = sc.overridden(stack)
    m.set_catchment_parameter(2, over)
    kernels = launched(m.run_cells)
    assert_path("D parameter table", stack, kernels, sc.step_kernels(stack, 15, table=True), n, sc.run_cells_chunks(T))
    gm = geo_matrix(geo)
    f = forcing(m)
    pset = (gm[:, 4] == 2).astype(np.int32)
    want = Expected(oracle, stack, gm, np.stack([sc.DEFAULT[stack], over]), f, st0, ta, rows_of(T, (128, 129)), pset=pset)
    check_cells(m, stack, want, slice(None), f"{stack} override")
    s_over = m.get_states()
    # the table kernels with the region set everywhere, then the UPAR kernels: the same bits
    m.set_catchment_parameter(2, sc.DEFAULT[stack])
    m.revert_to_initial_state()
    m.run_cells()
    table = {name: m.response(name) for name in sc.responses(stack)}, m.get_states()
    m.remove_catchment_parameter(2)
    m.revert_to_initial_state()
    kernels = launched(m.run_cells)
    upar = stack in ("pt_gs_k", "pt_hs_k", "hbv_stack")
    assert_path("D UPAR" if upar else "D no override", stack, kernels, sc.step_kernels(stack, 15, table=not upar), n, sc.run_cells_chunks(T))
    plain = Expected(oracle, stack, gm, sc.DEFAULT[stack], f, st0, ta, rows_of(T))
    check_cells(m, stack, plain, slice(None), f"{stack} region set")
    assert np.all(np.any(s_over[pset == 1] != plain.state[pset == 1], axis=1)), "the override must change every overridden cell"
    for name, v in table[0].items():
        same(m.response(name), v, f"{stack} table kernels vs UPAR {name}")
    same(m.get_states(), table[1], f"{stack} table kernels vs UPAR end state")
    note("D parameter table", f"{stack}: override on every third lane bit-identical; catchment sums {check_sums(m, stack):.3f}")


# ---- E: the calculation filter under the time split -----------------------------------------------------------------------------------
@pytest.mark.parametrize("stack", sc.STACKS)
def test_calculation_filter(sb, oracle, stack):
    n, T = 96, 200
    m, geo, ta, _ = region(sb, stack, n, T, cids=interleaved(n), cfg=14)
    st0 = initial_state(m, stack, n)
    m.set_states(st0)
    m.set_state_collection(-1, True)
    m.set_catchment_calculation_filter([2])
    kernels = launched(m.run_cells)
    assert_path("E filter", stack, kernels, sc.step_kernels(stack, 15, table=False), n, sc.run_cells_chunks(T))
    gm = geo_matrix(geo)
    on = gm[:, 4] == 2
    f = forcing(m, np.flatnonzero(on))
    want = Expected(oracle, stack, gm[on], sc.DEFAULT[stack], f, st0[on], ta, rows_of(T, (128, 129)))
    check_cells(m, stack, want, on, f"{stack} filtered, active cells")
    same(m.get_states()[~on], st0[~on], f"{stack} filtered-out state")
    for name in sc.responses(stack):
        assert np.all(np.isnan(m.response(name)[:, ~on])), name
    ids = m.catchment_ids
    k_on = int(np.flatnonzero(ids == 2)[0])
    for k in range(len(ids)):
        if k != k_on:
            assert np.all(m.catchment_discharges()[:, k] == 0.0) and np.all(m.catchment_charges()[:, k] == 0.0), ids[k]
    note("E filter", f"{stack}: every third lane stepped; catchment sums {check_sums(m, stack, [k_on]):.3f}")


# ---- F: collector modes ---------------------------------------------------------------------------------------------------------------
MODES = dict(pt_gs_k=tuple(range(16)), pt_hs_k=(0, 1, 4, 8, 15), hbv_stack=(0, 1, 4, 8, 15), pt_ss_k=(0, 1, 4, 8, 15), pt_hps_k=(0, 1, 4, 8, 15))


@pytest.mark.parametrize("stack", sc.STACKS)
def test_collector_modes(sb, oracle, stack):
    n, T = 100, 129
    m, geo, ta, _ = region(sb, stack, n, T, cfg=15)
    st0 = initial_state(m, stack, n)
    gm = geo_matrix(geo)
    want = Expected(oracle, stack, gm, sc.DEFAULT[stack], forcing(m), st0, ta, rows_of(T))
    _, _, full_series = oracle_run(oracle, stack, gm, sc.DEFAULT[stack], forcing(m), st0, ta)
    state_names = sb.capi.STATE_SERIES_NAMES[sc.STACK_ID[stack]]
    ref = None
    for mode in MODES[stack]:
        m.set_states(st0)
        m._ck(m._L.sb2_set_collector_mode(m._h, C.c_int(mode)))
        if stack == "pt_gs_k":
            assert_path(f"F mode {mode}", stack, launched(m.run_cells), sc.step_kernels(stack, mode, table=False), n, [T])
        else:
            m.run_cells()
        for name in sc.responses(stack):
            if mode & sc.collect_bit(name):
                same(m.response(name), want.resp[name], f"{stack} mode {mode} {name}")
            else:
                with pytest.raises(RuntimeError, match="not collected"):
                    m.response(name)
        if mode & 8:
            for r, d in want.rows.items():
                for name, v in d.items():
                    same(m.state_series(name, r, 1)[0], v, f"{stack} mode {mode} state series {name} row {r}")
            for name, v in (full_series or {}).items():
                same(m.state_series(name), v, f"{stack} mode {mode} state series {name}")
        else:
            with pytest.raises(RuntimeError, match="not collected"):
                m.state_series(state_names[0])
        now = (m.catchment_discharges(), m.catchment_charges(), m.get_states())
        same(now[2], want.state, f"{stack} mode {mode} end state")
        if ref is None:
            ref = now
        for a, b, what in zip(now, ref, ("discharges", "charges", "end state")):
            same(a, b, f"{stack} mode {mode} catchment {what} vs mode {MODES[stack][0]}")
    if stack != "pt_gs_k":
        note("F modes", f"{stack}: modes {MODES[stack]} (one kernel, collect read at run time)")


# ---- G, H, I: the pt_gs_k calibration batch ---------------------------------------------------------------------------------------------
def _perturbed(rng, k):
    P = np.tile(PTGSK_DEFAULT, (k, 1))
    P[:, 0] = rng.uniform(-3.0, -1.9, k)      # kirchner.c1
    P[:, 1] = rng.uniform(0.8, 0.99, k)       # c2
    P[:, 2] = rng.uniform(-0.15, -0.05, k)    # c3
    P[:, 4] = rng.uniform(-2.0, 2.0, k)       # tx
    P[:, 16] = rng.uniform(0.8, 1.4, k)       # p_corr
    return P


def ptgsk_optimizer(sb, n, T, cells_per_catchment):
    from shyft_b200 import synthetic
    geo, ta, env = synthetic.make_region(n, T, 9, config_index=4, cells_per_catchment=cells_per_catchment, start=1425168000)  # 2015-03-01
    m = sb.PTGSKOptModel(geo, PTGSK_DEFAULT)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    st0 = synthetic.default_state(0, n)
    m.set_states(st0)
    m.run_cells()
    obs = m.catchment_discharges()[:, :2].sum(axis=1).reshape(-1, 24).mean(axis=1)
    return m, geo, ta, st0, obs, sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, DAY, [1, 2], 1.0, 0)])


G_SHAPE = (240, 24 * 60, 2000)   # 8 step groups x 2 000 members = 16 000: exactly at the threshold, not split


def test_ptgsk_batch_unsplit_in_odd_chunks(sb, oracle):
    n, T, E = G_SHAPE
    ps = sc.ptgsk_batch_steps(n, T, E)
    chunks = [min(ps, T - d) for d in range(0, T, ps)]
    assert ps == 223 and chunks == [223] * 6 + [102]
    assert not sc.time_split(n, E) and sc.time_split(n, 1)
    m, geo, ta, st0, obs, opt = ptgsk_optimizer(sb, n, T, 80)
    P = _perturbed(np.random.default_rng(23), E)
    batch = []
    kernels = launched(lambda: batch.append(opt.calculate_goal_function_batch(P)))
    batch = batch[0]
    assert_path("G batch unsplit", "pt_gs_k", kernels, sc.step_kernels("pt_gs_k", 0, table=True), n, chunks, members=E)
    terms = [g for k, g in kernels if k.startswith("ptgsk_forcing_terms")]
    if all(g is not None for g in terms):   # grid.y of the forcing-terms kernel: the chunk in blocks of 8 steps
        assert [g[1] for g in terms] == [sc.ceil_div(c, 8) for c in chunks], terms
    one = []
    kernels = launched(lambda: one.append(opt.calculate_goal_function_batch(P[:1])))
    assert_path("G batch of one (split)", "pt_gs_k", kernels, sc.step_kernels("pt_gs_k", 0, table=True), n, [T], members=1)
    for i in (0, 999, 1999):
        assert batch[i] == opt.calculate_goal_function(P[i]), i
    assert one[0][0] == batch[0]
    f = forcing(m)
    gm = geo_matrix(geo)
    sel = np.isin(gm[:, 4], [1, 2])
    run = oracle.ptgsk_run_cells(gm, P[0], f, st0, ta.start * 10**6, H, ncore=8)
    want = oracle.nash_sutcliffe(obs, oracle.average_to_axis(run["avg_discharge"][:, sel].sum(axis=1), H, 0, 24, obs.size))
    assert batch[0] == pytest.approx(want, rel=1e-9)
    note("G batch unsplit", f"members 0 / 999 / 1999 = single evaluation; chunks of {ps} steps")


def test_ptgsk_batch_in_two_passes(sb):
    n, T, E = 64, 96, 65537
    m, geo, ta, st0, obs, opt = ptgsk_optimizer(sb, n, T, 32)
    P = _perturbed(np.random.default_rng(29), E)
    ps = sc.ptgsk_batch_steps(n, T, E)
    per_pass = 4 * sc.ceil_div(T, ps) + 1   # (forcing terms, snow, response, catchment reduction) per chunk, then the goal kernel
    k0 = m.kernel_launches()
    batch = opt.calculate_goal_function_batch(P)
    assert m.kernel_launches() - k0 == 2 * per_pass
    for i in (0, 65534, 65535, 65536):
        assert batch[i] == opt.calculate_goal_function(P[i]), i
    note("H batch in two passes", f"65 537 sets in 2 passes of {per_pass} launches (chunks of {ps} steps); members at the pass edge = single")


def test_red_zones_stay_intact_in_an_unsplit_ptgsk_batch():
    """case G under SB2_GUARD: the per-member scratch stride ps * n and the partial-sum stride are where an overrun would land"""
    env = dict(os.environ, SB2_GUARD="1")
    n, T, E = G_SHAPE
    prog = f"""
import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
import numpy as np
import shyft_b200 as sb
from shyft_b200 import capi
from test_gpu_step_paths import _perturbed, ptgsk_optimizer
m, geo, ta, st0, obs, opt = ptgsk_optimizer(sb, {n}, {T}, 80)
P = _perturbed(np.random.default_rng(23), {E})
g = opt.calculate_goal_function_batch(P)
assert np.all(np.isfinite(g)) and g[7] == opt.calculate_goal_function(P[7])
v, msg = capi.check_guards()
print('batch ok', 'guards', v, msg)
sys.exit(1 if v else 0)
"""
    r = subprocess.run([sys.executable, "-c", prog], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "batch ok" in r.stdout and "guards 0" in r.stdout
    note("I red zones", f"{E} members x {n} cells under SB2_GUARD: guards intact")


# ---- J: slot layouts --------------------------------------------------------------------------------------------------------------------
def slot_layout(n=300):
    cid = np.empty(n, dtype=np.int64)
    cid[:32] = 1 + np.arange(32) % 3       # interleaved lane by lane
    cid[5] = 99                            # a catchment of one cell
    cid[32:192] = 50                       # one catchment over five whole warps
    cid[192:] = 90 - np.arange(n - 192) // 6   # ids descending in runs of 6 cells, across warp boundaries
    return cid


@pytest.mark.parametrize("stack", ["pt_gs_k", "pt_hs_k"])
def test_slot_layouts(sb, stack):
    n, T = 300, 129
    m, geo, ta, _ = region(sb, stack, n, T, cids=slot_layout(n), cfg=16)
    m.set_states(initial_state(m, stack, n))
    m.run_cells()
    assert m.number_of_catchments() == 5 + 18
    note("J slot layouts", f"{stack}: 1-cell, 5-warp, interleaved and descending catchments; catchment sums {check_sums(m, stack):.3f}")
