"""Secondary measurements (not the bench.py line): BASELINE configs 3 and 5 on one GPU, reduced where a full run would take
minutes; prints one JSON line per config.  Usage: python tools/bench_configs.py [3] [5]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import shyft_b200 as sb
from shyft_b200 import synthetic

PTGSK = [-2.439, 0.966, -0.10, 1.5, -0.5, 2.0, 0.1, 1.0, 5.0, 5.0, 30.0, 0.9, 0.6, 5.0, 0.4, 0.4, 1.0, 0.0, 0.0, 0.2, 1.26, 0.04, 100.0, 0.0, 6.0, 1.0, 7.0, 0.0,
         221.0, 0.0, 1.0]
PTHSK = [-2.439, 0.966, -0.10, 1.5, 0.1, 0.0, 1.0, 0.0, 0.5, 6.0, 1.0, 0.2, 1.26, 1.0, 7.0, 0.0, 0.0, 1.0]
PTHPSK = [-2.439, 0.966, -0.10, 1.5, 0.1, 0.0, 0.5, 2.0, 1.0, 30.0, 0.9, 0.6, 5.0, 5.0, 5.0, 0.0, 6.0, 1.0, 0.2, 1.26, 1.0, 7.0, 0.0, 1.0]
HBV = [300.0, 2.0, 150.0, 25.0, 0.5, 0.3, 0.8, 0.02, 0.1, 0.0, 1.0, 0.0, 0.5, 1.0, 0.2, 1.26, 6.0, 1.0, 7.0, 0.0, 0.0, 1.0]
which = [int(a) for a in sys.argv[1:]] or [3, 5]


def timed(fn, reps=2):
    fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) / 1000.0)
    return best


if 3 in which:  # pt_hs_k and hbv_stack, 400k cells x 5 years hourly, river routing (windowed: the axis cannot be resident)
    n, years = 400000, float(os.environ.get("SB2_C3_YEARS", "1"))
    T = int(8760 * years)
    geo, ta, env = synthetic.make_region(n, T, 64, config_index=2, with_routing=True)
    rivers = synthetic.river_chain(n // 1000, depth=8)
    for name, cls, sid, nbytes in (("pt_hs_k", sb.PTHSKOptModel, 1, 56), ("hbv_stack", sb.HbvStackOptModel, 2, 56), ("pt_ss_k", sb.PTSSKOptModel, 3, 56),
                                   ("pt_hps_k", sb.PTHPSKOptModel, 4, 56)):
        m = cls(geo)
        m.initialize_cell_environment(ta)
        m._set_sources(env)
        m.set_states(synthetic.default_state(sid, n))
        m.set_river_network(rivers)
        ip = sb.InterpolationParameter()

        def run():
            m.revert_to_initial_state() if run.n else None
            run.n += 1
            m.run_windowed(ip, window_steps=int(os.environ.get("SB2_C3_WINDOW", "1024")))
            m.river_output_flow_m3s(8)
        run.n = 0
        s = timed(run)
        step_ms, interp_ms = m.last_run_kernel_ms()
        print(json.dumps({"config": 3, "stack": name, "cells": n, "steps": T, "seconds": s, "cell_steps_per_s": n * T / s,
                          "step_kernel_cell_steps_per_s": n * T / (step_ms / 1e3), "step_kernel_GBps_at_56B": 56 * n * T / (step_ms / 1e3) / 1e9,
                          "interp_ms": interp_ms, "step_ms": step_ms}))
        del m

if 5 in which:  # calibration ensemble: parameter sets x 10k-cell catchment x 3 years hourly, NSE goal
    # under torchrun (python -m torch.distributed.run --nproc-per-node N tools/bench_configs.py 5) the population is sharded over the
    # ranks, every rank holds all cells; the only exchange is one all_gather of the goal values (shyft_b200/sharding.py)
    import torch.distributed as dist
    from shyft_b200 import sharding
    world, rank, local_rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # SB2_C5_STACK: pt_gs_k (default), pt_hs_k, hbv_stack or pt_hps_k -- the stacks whose batch runs as grid layers on the device
    stack = os.environ.get("SB2_C5_STACK", "pt_gs_k")
    # SB2_C5_TARGET=routed: the target is the routed outflow of river 8, the outlet of a chain of eight (synthetic.river_chain over the
    # 10 catchments), and every set also draws its own routing velocity
    routed = os.environ.get("SB2_C5_TARGET", "discharge") == "routed"
    n, T, sets = 10000, 26280, int(os.environ.get("SB2_C5_SETS", "256"))
    geo, ta, env = synthetic.make_region(n, T, 64, config_index=4, with_routing=routed)
    cls, par, sid = {"pt_gs_k": (sb.PTGSKOptModel, PTGSK, 0), "pt_hs_k": (sb.PTHSKOptModel, PTHSK, 1), "hbv_stack": (sb.HbvStackOptModel, HBV, 2),
                     "pt_hps_k": (sb.PTHPSKOptModel, PTHPSK, 4)}[stack]
    m = cls(geo, par, device=local_rank)
    m.run_interpolation(sb.InterpolationParameter(), ta, env)
    m.set_states(synthetic.default_state(sid, n))
    if routed:
        m.set_river_network(synthetic.river_chain(10))
    m.run_cells()
    if routed:
        obs = m.river_output_flow_m3s(8).reshape(-1, 24).mean(axis=1)
        opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, 86400, [], 1.0, 0, catchment_property=3, river_id=8)])
    else:
        obs = m.catchment_discharges().sum(axis=1).reshape(-1, 24).mean(axis=1)
        opt = sb.Optimizer(m, [sb.TargetSpecification(obs, ta.start, 86400, list(range(1, 11)), 1.0, 0)])
    rng = np.random.default_rng(5)
    P = np.tile(par, (sets, 1))
    if stack == "pt_gs_k":
        P[:, 0] = rng.uniform(-3.0, -1.9, sets); P[:, 1] = rng.uniform(0.8, 0.99, sets); P[:, 2] = rng.uniform(-0.15, -0.05, sets)
        P[:, 3] = rng.uniform(0.5, 2.5, sets); P[:, 4] = rng.uniform(-2, 2, sets); P[:, 5] = rng.uniform(1, 4, sets)
        P[:, 14] = rng.uniform(0.2, 0.8, sets); P[:, 16] = rng.uniform(0.8, 1.4, sets)
    elif stack == "pt_hs_k":   # c1, c2, c3, ae_scale, tx, cx, p_corr
        P[:, 0] = rng.uniform(-3.0, -1.9, sets); P[:, 1] = rng.uniform(0.8, 0.99, sets); P[:, 2] = rng.uniform(-0.15, -0.05, sets)
        P[:, 3] = rng.uniform(0.5, 2.5, sets); P[:, 5] = rng.uniform(-2, 2, sets); P[:, 6] = rng.uniform(0.5, 2.0, sets)
        P[:, 10] = rng.uniform(0.8, 1.4, sets)
    elif stack == "pt_hps_k":  # c1, c2, c3, ae_scale, tx, wind_scale, fast / slow albedo decay rate, p_corr
        P[:, 0] = rng.uniform(-3.0, -1.9, sets); P[:, 1] = rng.uniform(0.8, 0.99, sets); P[:, 2] = rng.uniform(-0.15, -0.05, sets)
        P[:, 3] = rng.uniform(0.5, 2.5, sets); P[:, 5] = rng.uniform(-2, 2, sets); P[:, 7] = rng.uniform(1.0, 3.0, sets)
        P[:, 12] = rng.uniform(2.0, 8.0, sets); P[:, 13] = rng.uniform(2.0, 8.0, sets); P[:, 17] = rng.uniform(0.8, 1.4, sets)
    else:                      # fc, beta, lp, uz1, kuz2, kuz1, perc, klz, tx, p_corr
        P[:, 0] = rng.uniform(150, 450, sets); P[:, 1] = rng.uniform(1, 4, sets); P[:, 2] = rng.uniform(100, 200, sets)
        P[:, 3] = rng.uniform(10, 40, sets); P[:, 4] = rng.uniform(0.2, 0.7, sets); P[:, 5] = rng.uniform(0.1, 0.4, sets)
        P[:, 6] = rng.uniform(0.4, 1.2, sets); P[:, 7] = rng.uniform(0.01, 0.05, sets); P[:, 9] = rng.uniform(-2, 2, sets)
        P[:, 13] = rng.uniform(0.8, 1.4, sets)
    if routed:
        off = {"pt_gs_k": 25, "pt_hs_k": 13, "hbv_stack": 17, "pt_hps_k": 20}[stack]   # routing.velocity
        P[:, off] = par[off] * rng.uniform(0.5, 1.5, sets)
    b, e = sharding.partition_parameter_sets(sets, world, rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g_local = opt.calculate_goal_function_batch(P[b:e])
    g = sharding.gather_goal_values(g_local, sets, device=torch.device("cuda", local_rank) if world > 1 else None)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    if world > 1:
        t_all = torch.tensor([s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
        s = float(t_all.item())
        if rank != 0:
            dist.barrier(); dist.destroy_process_group(); sys.exit(0)
    t0 = time.perf_counter()
    g1 = np.array([opt.calculate_goal_function(p) for p in P[:8]])
    s1 = (time.perf_counter() - t0) / 8
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local_rank)], capture_output=True,
                         text=True).stdout.strip()
    print(json.dumps({"config": 5, **({} if stack == "pt_gs_k" and not routed else {"stack": stack, "gpu": gpu}),
                      **({"target": "routed"} if routed else {}), "n_gpus": world, "sets": sets, "cells": n, "steps": T, "batch_seconds": s, "cell_steps_per_s": sets * n * T / s,
                      "one_at_a_time_seconds_per_set": s1, "cell_steps_per_s_one_at_a_time": n * T / s1, "batch_equals_single": bool(np.array_equal(g[:8], g1)),
                      "best_goal": float(g.min()), "extrapolated_4096_sets_seconds": s * 4096 / sets}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
