#!/usr/bin/env python
"""bench.py -- cell-timesteps/s of the pt_gs_k run_cells hot path (BASELINE.json), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--cells C] [--years Y] [--window S] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the CPU path (oracle port; the real reference cannot be built here)

A "step" is one pass of the hot path over the whole workload: BASELINE configs[1], pt_gs_k, 100 000 cells x 10 years
hourly (87 600 steps), BTK temperature + IDW for the other four variables, discharge collector (56 algorithmic bytes
per cell-step), run window by window because the [time][cell] forcing (350 GB) cannot be resident.  At N > 1 the workload is
BASELINE configs[3]: ONE region of 1 000 000 cells x 10 years sharded over the N ranks (1 000 000 / N cells per GPU -- total work
fixed, "strong" scaling; --cells C overrides with C cells per GPU), the per-catchment discharge series of the shards placed at
their global catchment index and summed across ranks with NCCL; the reduced [T][n_catchments] tensor is what the end-to-end
leg copies back, and rank 0 re-computes one straddling catchment on its own to check it.

  value     cell-steps / device time with the station series already in HBM (CUDA events on the launching stream)
  e2e       same metric through the public API with HOST buffers: station series + states H2D (pinned memory),
            catchment discharge + end states D2H, inside the timed region
  roofline  the step kernel alone: 56 B x cell-steps / its CUDA-event time vs the measured HBM copy peak
  cpu_baseline  the CPU oracle's threaded run_cells on a bounded sample, same inputs, rank 0 only
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (no __pycache__)

BYTES_PER_CELL_STEP = 56  # 5 forcings read + avg_discharge, charge_m3s written (BASELINE.md section 3)
NCU_PROFILE = os.path.join(ROOT, "profiles", "ncu_pipeline_r02_shipped.json")  # tools/ncu_pipeline_json.py of the shipped configuration
DUMP_BYTES = 60 * 10**6   # --dump-outputs: data budget, so that the files with their .npy headers stay under 64 MB
DUMP_SEED = 20260101
PTGSK_DEFAULT = [-2.439, 0.966, -0.10, 1.5, -0.5, 2.0, 0.1, 1.0, 5.0, 5.0, 30.0, 0.9, 0.6, 5.0, 0.4, 0.4, 1.0, 0.0, 0.0, 0.2, 1.26, 0.04, 100.0, 0.0,
                 6.0, 1.0, 7.0, 0.0, 221.0, 0.0, 1.0]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cells", type=int, default=0, help="cells per GPU (default: 100 000 on one GPU = configs[1]; 1 000 000 / N on N GPUs = configs[3])")
    ap.add_argument("--years", type=float, default=10.0)
    ap.add_argument("--stations", type=int, default=64)
    ap.add_argument("--window", type=int, default=4096, help="time steps per forcing window (round 2, with one launch set per window: 2048 -> 9.54, 4096 -> 9.62 G cell-steps/s)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU work of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle legs (cpu_baseline and config.parity_check)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (catchment discharge and charge series, end states) as DIR/<name>.npy, "
                         "float64; above %d MB together every array keeps the same seeded sample of its rows" % (DUMP_BYTES // 10**6))
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    a.cells_given = a.cells > 0
    if not a.cells_given:
        a.cells = 100000 if world == 1 else 1000000 // world
    # window buffers: keep cells x window at what 100 000 cells x 4 096 steps take (33 GB of forcing + series and 16 GB of scratch per GPU)
    a.window = max(256, min(a.window, (a.window * 100000 // a.cells) // 64 * 64))
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_workload(args, rank, world):
    from shyft_b200 import synthetic
    n_steps = int(round(args.years * 8760))
    n_total = args.cells * world
    # the whole region is generated identically on every rank; each rank keeps its shard (cells are independent)
    # catchments of 1 000 cells; at N > 1 of 1 500 cells, so that catchments straddle the shard boundaries and the all-reduce has real sums to form
    geo, ta, env = synthetic.make_region(n_total, n_steps, args.stations, config_index=1, cells_per_catchment=1000 if world == 1 else 1500)
    from shyft_b200.sharding import partition_cells
    b, e = partition_cells(n_total, world, rank)
    return geo, geo[b:e], ta, env, synthetic.default_state(0, e - b)


def pinned_copy(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
    v = t.numpy()
    v[...] = a
    return v, t


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write each array of `arrays` as out_dir/<name>.npy in float64.  When they take more than `budget` bytes together, every array
    keeps the same fraction of its rows (axis 0), drawn with a fixed seed and kept in order, so that two runs with the same arguments
    write the same rows.  -> {name: [rows written, rows computed]}"""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    frac = min(1.0, budget / max(1, sum(a.nbytes for a in arrays.values())))
    kept = {}
    for name, a in arrays.items():
        k = max(1, int(a.shape[0] * frac))
        if k < a.shape[0]:
            a = a[np.sort(np.random.default_rng(DUMP_SEED).choice(a.shape[0], k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        kept[name] = [int(a.shape[0]), int(arrays[name].shape[0])]
    return kept


FORCING = ("temperature", "precipitation", "radiation", "wind_speed", "rel_hum")


def oracle_pass(O, gm, ta, env, window, cores, n_steps=None):
    """One pass of the hot path on the CPU oracle, the way the device runs it: per window of `window` steps interpolate()
    (BTK temperature + IDW, core/region_model.h:397-527) and run_cells (:578-597, the reference's work-queue threading, :991-1021) with the
    state carried from window to window, over the whole time axis.  -> (seconds in interpolation, seconds in run_cells, end state)"""
    n = gm.shape[0]
    T = ta.n if n_steps is None else n_steps
    dt_us = ta.delta_t * 10**6
    st = np.tile(np.array([0.4, 0.1, 30000.0, 1.26, 0.0, 0.0, 0.0, 0.0, 0.8]), (n, 1))
    t_interp = t_run = 0.0
    for w0 in range(0, T, window):
        wn = min(window, T - w0)
        t0_us = (ta.start + w0 * ta.delta_t) * 10**6
        a = time.perf_counter()
        f = {}

        def one(name):
            xyz, vals = getattr(env, name)
            vals = O.average_accessor_same_axis(vals[w0:w0 + wn], dt_us)
            if name == "temperature":   # btk_interpolation: one thread (core/bayesian_kriging.h:280-402 has no threading of its own)
                f[name] = O.btk_run(xyz, vals, gm[:, :3], t0_us, dt_us)
            else:                       # idw::run_interpolation splits the cells over ncore threads (core/inverse_distance.h:503-560)
                f[name] = O.idw_run(name, xyz, vals, gm[:, :3], O.idw_par(max_members=20 if name == "precipitation" else 10), dst_slope=gm[:, 5],
                                    ncore=cores)
        # the five variables are interpolated by five concurrent tasks, as region_model::interpolate launches them (core/region_model.h:456-523);
        # the oracle's C functions release the GIL
        tasks = [threading.Thread(target=one, args=(name,)) for name in FORCING]
        for t in tasks:
            t.start()
        for t in tasks:
            t.join()
        b = time.perf_counter()
        st = O.ptgsk_run_cells(gm, PTGSK_DEFAULT, f, st, t0_us, dt_us, collect_response=False, ncore=cores)["state"]
        c = time.perf_counter()
        t_interp += b - a
        t_run += c - b
    return t_interp, t_run, st


def cpu_baseline(args, geo_local, ta, env, target_seconds):
    """The CPU oracle on a bounded sample of the SAME workload: cells evenly spread over the shard, the whole time axis, window by
    window with interpolation (see oracle_pass).  `value` = cell-steps / (interpolation + run_cells) -- the same pass the device
    is timed on; the run_cells-only rate is reported beside it.  Sized from a short probe so that one pass takes ~target_seconds."""
    from oracle import oracle as O
    cores = O.hardware_concurrency()
    T = ta.n

    def sample(n):
        idx = np.linspace(0, geo_local.shape[0] - 1, n).astype(np.int64)  # spread over the shard: all elevations / climates
        return O.geo_matrix(geo_local[idx])

    n_probe = max(64, 8 * cores)
    ti, tr, _ = oracle_pass(O, sample(n_probe), ta, env, args.window, cores, n_steps=min(T, 2 * args.window))   # probe: two windows
    rate = n_probe * min(T, 2 * args.window) / (ti + tr)
    n = int(min(geo_local.shape[0], max(n_probe, rate * target_seconds / T)))
    ti, tr, _ = oracle_pass(O, sample(n), ta, env, args.window, cores)
    return {"value": n * T / (ti + tr), "unit": "cell-timesteps/s", "cores": cores, "kind": "port",
            "run_cells_only_value": n * T / tr, "interpolation_share": ti / (ti + tr),
            "sample_cells": n, "sample_fraction_of_cells": n / float(geo_local.shape[0]), "extrapolated": True,
            "sample": f"{n} of {geo_local.shape[0]} cells (evenly spread over the shard) x all {T} steps, window by window ({args.window} steps) with "
                      f"BTK + IDW interpolation and the state carried over, oracle with {cores} threads, one pass: interpolation {ti:.2f} s + run_cells {tr:.2f} s"}


def parity_check(sb, args, geo, ta, env):
    """The end-to-end census of tests/test_gpu_e2e_parity.py on a small slice of THIS workload, through the path timed above (dense DMMA
    interpolation -> step kernels, window by window) against the oracle's interpolate -> run_cells: 256 cells (16 runs of 16 neighbours
    spread over the shard) x the first year.  Reported under config.parity_check."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from e2e_cases import oracle_forcing, run_device_windows
    from e2e_census import Census
    from oracle import oracle as O
    from shyft_b200 import synthetic
    T = min(ta.n, 8760)
    starts = np.linspace(0, geo.shape[0] - 16, 16).astype(np.int64) // 16 * 16
    g = geo[(starts[:, None] + np.arange(16)[None, :]).ravel()]
    ta1 = sb.TimeAxis(ta.start, ta.delta_t, T)
    env1 = sb.RegionEnvironment(**{k: (getattr(env, k)[0], getattr(env, k)[1][:T]) for k in FORCING})
    gm, f = oracle_forcing(O, g, ta1, env1, btk_temperature=True, ncore=O.hardware_concurrency())
    st0 = synthetic.default_state(0, g.shape[0])
    want = O.ptgsk_run_cells(gm, PTGSK_DEFAULT, f, st0, ta1.start * 10**6, ta1.delta_t * 10**6, collect_response=True, collect_state=True,
                             ncore=O.hardware_concurrency())
    want.pop("state")
    m = sb.PTGSKModel(g, PTGSK_DEFAULT)
    m.set_state_collection(-1, True)
    m.initialize_cell_environment(ta1)
    m._set_sources(env1)
    m.set_states(st0)
    cs = Census(want, f, tx=PTGSK_DEFAULT[4])
    run_device_windows(m, sb.InterpolationParameter(), T, args.window, ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow"),
                       sb.capi.STATE_SERIES_NAMES[sb.PT_GS_K], cs.add_window)
    c = cs.result()
    return {"slice": f"{g.shape[0]} cells x {T} steps of this workload, device run_windowed vs oracle interpolate + run_cells, rtol 1e-9",
            "cell_steps_within_1e-9": c["cell_steps_within"], "cells_with_a_decision_flip": c["cells_with_a_decision_flip"],
            "flip_rate_per_cell_year": c["flip_rate_per_cell_year"], "first_divergence_by_cause": c["first_divergence_by_cause"],
            "forcing_worst_rel": max(c["forcing_worst_rel"].values()), "discharge_within": c["series"]["avg_discharge"]["within"],
            "full_census": "tests/test_gpu_e2e_parity.py (2 048 cells x 2 years; DESIGN.md section 2)"}


def workload_name(args, n, T, world=1):
    region = f"{n} cells" if world == 1 else f"{n * world} cells sharded over {world} GPUs ({n} per GPU)"
    return (f"pt_gs_k {region} x {T} hourly steps ({args.years:g} y), BTK temperature + IDW precipitation/radiation/wind/rel_hum, "
            f"{args.stations} stations, discharge collector, windows of {args.window} steps")


def run_reference(args):
    """--impl reference: the reference's CPU path for the same pass.  The reference itself cannot be built here (DESIGN.md), so this is the
    oracle port with all host threads; each step is one oracle_pass over the whole axis on a bounded sample of the cells."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    geo, geo_local, ta, env, st0 = build_workload(args, 0, 1)
    vals, last = [], None
    per_pass = max(4.0, min(args.cpu_seconds, 150.0 / (args.warmup + args.steps)))   # the whole run stays within a few minutes
    for i in range(args.warmup + args.steps):
        last = cpu_baseline(args, geo_local, ta, env, per_pass)
        if i >= args.warmup:
            vals.append(last["value"])
    v = statistics.mean(vals)
    n_steps = ta.n
    last["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": "cell-timesteps/sec (pt_gs_k run_cells)", "value": v, "unit": "cell-timesteps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * args.cells * world * n_steps / v, "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args, args.cells, n_steps, world), "cells_per_gpu": args.cells, "n_steps": n_steps,
                   "window_steps": args.window, "extrapolated": True, "sample_fraction_of_cells": last["sample_fraction_of_cells"],
                   "note": "CPU arm = the oracle PORT of the reference's algorithm (kind: port; the reference needs boost 1.68 / armadillo / dlib and "
                           "cannot be built here): interpolation + run_cells window by window over the WHOLE time axis on a sample of the cells, all "
                           "host threads; ms_per_step is the sample's rate extrapolated to the whole workload.  The port evaluates gamma_p / lgamma "
                           "in full double where the reference uses boost's reduced-precision policies, so it is somewhat slower than real Shyft "
                           "in the snow routine."},
        "cpu_baseline": last,
        "e2e": {"value": v, "unit": "cell-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import shyft_b200 as sb
    from shyft_b200 import sharding

    geo_all, geo, ta, env, st0 = build_workload(args, rank, world)
    n, T = geo.shape[0], ta.n
    _, global_cids = sharding.global_catchment_index(geo_all["catchment_id"])
    m = sb.PTGSKOptModel(geo, PTGSK_DEFAULT, device=local_rank)
    ip = sb.InterpolationParameter()  # BTK temperature + IDW (defaults of core/region_model.h:65-95)
    # host buffers of the end-to-end leg live in pinned memory
    keep = []
    env_pinned = sb.RegionEnvironment()
    for name in sb.capi.FORCING_NAMES:
        xyz, vals = getattr(env, name)
        v, t = pinned_copy(vals)
        keep.append(t)
        setattr(env_pinned, name, (xyz, v))
    st_pinned, t = pinned_copy(st0)
    keep.append(t)
    # results of the end-to-end leg land in pinned memory too: the region's [T][n_catchments] discharge (at N > 1 the all-reduced GLOBAL
    # tensor, every rank copies it back) and this rank's end states
    n_catch_out = m.number_of_catchments() if world == 1 else int(global_cids.size)
    q_pinned, q_pinned_t = pinned_copy(np.zeros((T, n_catch_out)))
    keep.append(q_pinned_t)
    s_pinned, t = pinned_copy(np.zeros_like(st0))
    keep.append(t)
    h2d = sum(getattr(env, k)[1].nbytes + getattr(env, k)[0].nbytes for k in sb.capi.FORCING_NAMES) + st0.nbytes
    d2h = T * n_catch_out * 8 + st0.nbytes

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    reduced = {"q": None}

    def reduce_catchments():
        """the region's catchment discharge: this shard's sums at their global catchment index, summed over the ranks (NCCL)"""
        if world == 1:
            return None
        torch.cuda.nvtx.range_push("all_reduce catchment discharge")
        reduced["q"] = sharding.global_catchment_series(m, global_cids, "discharge")
        torch.cuda.nvtx.range_pop()
        return reduced["q"]

    def device_pass():
        m.revert_to_initial_state()
        m.run_windowed(ip, window_steps=args.window)
        reduce_catchments()

    e2e_parts = {}

    def e2e_pass():
        t = [time.perf_counter()]

        def lap(name):
            t.append(time.perf_counter())
            e2e_parts.setdefault(name, []).append(1000.0 * (t[-1] - t[-2]))
        m.initialize_cell_environment(ta); lap("initialize_cell_environment")
        m._set_sources(env_pinned); lap("set_sources_h2d")
        m.initial_state = st_pinned
        m.set_states(st_pinned); lap("set_states_h2d")
        m.run_windowed(ip, window_steps=args.window); lap("run_windowed")
        g = reduce_catchments(); lap("all_reduce")
        if g is None:
            m.catchment_discharges(out=q_pinned)
        else:
            q_pinned_t.copy_(g)          # device -> pinned host (synchronous for pinned destinations)
            torch.cuda.synchronize()
        m.get_states(out=s_pinned); lap("results_d2h")
        return q_pinned, s_pinned

    def timed(fn, k):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # resident-input leg
    m.initialize_cell_environment(ta)
    m._set_sources(env)
    m.set_states(st0)
    for _ in range(args.warmup):
        device_pass()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = m.kernel_launches()
    step_ms_acc, interp_ms_acc = [], []

    def device_pass_recorded():
        device_pass()
        s, i = m.last_run_kernel_ms()
        step_ms_acc.append(s)
        interp_ms_acc.append(i)

    total_ms = timed(device_pass_recorded, args.steps)
    launches = m.kernel_launches() - l0
    clocks = sampler.stop() if sampler else None
    cq_device = m.catchment_discharges() if world == 1 else reduced["q"].cpu().numpy()
    last_step = None
    if args.dump_outputs:
        # what a caller of the timed path receives from its last step; at N > 1 the region's all-reduced series and rank 0's end states
        last_step = {"catchment_discharge": cq_device,
                     "catchment_charge": m.catchment_charges() if world == 1 else
                     sharding.global_catchment_series(m, global_cids, "charge").cpu().numpy(),
                     "end_state": m.get_states()}
    chunk_steps = m.step_chunk_steps()
    # end-to-end leg (host buffers)
    e2e_pass()
    wall = []
    barrier()
    for _ in range(max(1, min(args.steps, 3))):
        t0 = time.perf_counter()
        cq_e2e, _ = e2e_pass()
        torch.cuda.synchronize()
        wall.append(time.perf_counter() - t0)
    e2e_s = torch.tensor([statistics.mean(wall)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    if not np.array_equal(cq_e2e, cq_device):
        raise SystemExit("bench.py: the end-to-end pass and the resident pass disagree")
    if not np.all(np.isfinite(cq_device)):
        raise SystemExit("bench.py: non-finite catchment discharge")
    multi_gpu_check = None
    if world > 1 and rank == 0:
        # rank 0 re-computes, on its own and from scratch, the catchment that straddles the boundary between shard 0 and shard 1 (all of its
        # cells, from both shards) over the first window, and compares with that column of the all-reduced tensor it just copied back
        gcix, _ = sharding.global_catchment_index(geo_all["catchment_id"])
        b0, e0 = sharding.partition_cells(geo_all.shape[0], world, 0)
        k = int(gcix[e0 - 1])
        cells = np.nonzero(gcix == k)[0]
        straddles = bool(cells.max() >= e0)
        Wc = min(args.window, T)
        mc = sb.PTGSKOptModel(geo_all[cells], PTGSK_DEFAULT, device=local_rank)
        mc.initialize_cell_environment(ta)
        mc._set_sources(env)
        mc.set_states(synthetic_state(cells.size))
        mc.run_windowed(ip, start_step=0, n_steps=Wc, window_steps=Wc)
        want = mc.catchment_discharges(0, Wc)[:, 0]
        got = cq_e2e[:Wc, k]
        err = float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-300)))
        if not err <= 1e-12:
            raise SystemExit(f"bench.py: the all-reduced discharge of catchment index {k} differs from its single-GPU recomputation (rel {err:.3e})")
        multi_gpu_check = {"catchment_index": k, "cells": int(cells.size), "straddles_shard_boundary": straddles, "steps": int(Wc), "max_rel_diff": err,
                           "what": "column of the all-reduced [T][n_catchments] tensor (as copied back by the end-to-end leg) vs the same catchment "
                                   "stepped alone on rank 0"}
        del mc

    if rank == 0:
        cell_steps = float(n) * T * world
        ms_per_step = total_ms / args.steps
        value = cell_steps / (ms_per_step / 1000.0)
        peak, peak_src = measured_peaks()
        k_ms = statistics.mean(step_ms_acc)  # rank 0's step kernels per pass
        achieved = BYTES_PER_CELL_STEP * float(n) * T / (k_ms / 1000.0) / 1e9
        chunk = max(1, min(chunk_steps if chunk_steps > 0 else args.window, args.window, T))
        n_launch_sets = sum((min(args.window, T - w0) + chunk - 1) // chunk for w0 in range(0, T, args.window))
        prof = json.load(open(NCU_PROFILE)) if os.path.exists(NCU_PROFILE) else None
        out = {
            "metric": "cell-timesteps/sec (pt_gs_k run_cells)", "value": value, "unit": "cell-timesteps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if (world == 1 or args.cells_given) else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args, n, T, world),
                       "cells_per_gpu": n, "n_steps": T, "window_steps": args.window, "step_chunk_steps": chunk,
                       "l2": "inputs larger than L2: every window streams %.0f MB of forcing + series per pass" % (n * args.window * 56 / 1e6),
                       "interp_ms_per_step": statistics.mean(interp_ms_acc), "step_kernel_ms_per_step": k_ms,
                       "scaling_note": None if world == 1 else (
                           "weak: --cells per GPU given" if args.cells_given else
                           "strong over N >= 2: BASELINE configs[3], one region of 1 000 000 cells sharded over the ranks; N = 1 runs configs[1] (100 000 cells)")},
            "e2e": {"value": cell_steps / float(e2e_s.item()), "unit": "cell-timesteps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "rank0_ms": {k: round(statistics.mean(v[1:]), 2) for k, v in e2e_parts.items()},
                    "result": "region catchment discharge [T][%d]%s + this rank's end states, into pinned host memory" % (
                        n_catch_out, "" if world == 1 else " (the NCCL all-reduced global tensor)")},
            "gpu_launches": int(launches),
            "clocks": clocks,
            # One launch = run_cells over one chunk of the forcing window: the three kernels of the phase pipeline back to back.  "achieved"
            # divides the ALGORITHMIC bytes (56 B per cell-step, BASELINE.md section 3) by their CUDA-event time, measured live on the
            # launching stream.  "traffic", the pipe utilisation and the instruction counts come from the ncu --set full capture of the SAME
            # configuration committed as profiles/ncu_pipeline_r02_shipped.json (tools/ncu_pipeline_json.py), scaled by cell-steps.
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (prof["dram_bytes_per_cell_step"] * n * chunk) if prof else None,
                         "kernel": "run_cells chunk = ptgsk_forcing_terms_kernel<1> + ptgsk_snow_kernel<0,1> + ptgsk_response_kernel<1,1>",
                         "launches_per_step": n_launch_sets, "avg_launch_ms": k_ms / n_launch_sets,
                         "algorithmic_bytes_per_launch": BYTES_PER_CELL_STEP * n * chunk, "peak_source": peak_src,
                         "binding_roof": None if not prof else {
                             "pipe": "fp64 issue / latency", "source": os.path.relpath(NCU_PROFILE, ROOT) + " (" + prof["report"] + ")",
                             "per_kernel": {k["kernel"]: {"share_of_ncu_time": round(k["ms"] / sum(q["ms"] for q in prof["kernels"]), 3),
                                                          "fp64_pipe_active_pct": round(k["fp64_pipe_active_pct"], 1),
                                                          "issue_active_pct": round(k["issue_active_pct"], 1),
                                                          "fp64_instructions_per_cell_step": round(k["fp64_instructions_per_cell_step"], 1),
                                                          "instructions_per_cell_step": round(k["instructions_per_cell_step"], 1),
                                                          "dram_bytes_per_cell_step": round(k["dram_bytes_per_cell_step"], 1)} for k in prof["kernels"]}},
                         "note": "fp64-compute bound, not HBM bound: 16-25 exp/log, an adaptive ODE step and incomplete gamma functions "
                                 "per cell-step against 56 bytes (DESIGN.md section 3, SURVEY H3)"},
        }
        if multi_gpu_check is not None:
            out["config"]["multi_gpu_check"] = multi_gpu_check
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"] = cpu_baseline(args, geo, ta, env, args.cpu_seconds)
            out["config"]["parity_check"] = parity_check(sb, args, geo, ta, env)
        if last_step is not None:
            out["config"]["dump_outputs"] = {"dir": args.dump_outputs, "rows_written_of": dump_outputs(args.dump_outputs, last_step)}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def synthetic_state(n):
    from shyft_b200 import synthetic
    return synthetic.default_state(0, n)


if __name__ == "__main__":
    main()
