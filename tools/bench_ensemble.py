"""Forcing-ensemble measurement (not the bench.py line): 51 members x 240 hourly steps of pt_gs_k and hbv_stack on 10 000 and 100 000
cells, temperature by Bayesian kriging over 64 stations and precipitation by IDW per member, radiation, wind and relative humidity
from deterministic sources.  Times RegionModel.run_ensemble against the member loop it replaces (set the member's sources, interpolate,
run_cells from the same state, read the catchment sums), each after a warm-up call, by a host clock around a call that ends in a
device sync.  The two are timed alternately `--repeats` times; the median and the spread (min, max) of each are reported.  Prints one JSON
line per case with the card and its power limit read in the same run.

Usage: python tools/bench_ensemble.py [--out FILE.jsonl] [--cells 10000,100000] [--stacks pt_gs_k,hbv_stack] [--members 51] [--repeats 7]"""
import argparse
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

MODELS = dict(pt_gs_k=(sb.PTGSKOptModel, 0), hbv_stack=(sb.HbvStackOptModel, 2))
NAMES = ("temperature", "precipitation", "radiation", "wind_speed", "rel_hum")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, limit = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout.strip() else ("?", "?")
    return name, limit


def case(stack, n, T, E, seed=0):
    geo, ta, env = synthetic.make_region(n, T, 64, config_index=1, cells_per_catchment=max(1, n // 10), start=1420070400)
    cls, sid = MODELS[stack]
    m = cls(geo)
    m.initialize_cell_environment(ta)
    m._set_sources(env)
    m.set_states(synthetic.default_state(sid, n))
    rng = np.random.default_rng(seed)
    members = []
    for _ in range(E):
        xt, vt = env.temperature
        xp, vp = env.precipitation
        members.append(sb.RegionEnvironment(temperature=(xt, vt + rng.normal(0.0, 1.0, size=(1, vt.shape[1])) + rng.normal(0.0, 0.2, size=vt.shape)),
                                            precipitation=(xp, vp * rng.uniform(0.6, 1.4, size=(1, vp.shape[1])))))
    return m, env, members


def member_loop(m, env, members, ip):
    st = m.get_states()
    q = []
    for e in members:
        full = sb.RegionEnvironment(**{k: getattr(e, k) if getattr(e, k) is not None else getattr(env, k) for k in NAMES})
        m.interpolate(ip, full, best_effort=False)
        m.set_states(st)
        m.run_cells()
        q.append(m.catchment_discharges())
    m.set_states(st)
    return np.array(q)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--cells", default="10000,100000")
    ap.add_argument("--stacks", default="pt_gs_k,hbv_stack")
    ap.add_argument("--members", type=int, default=51)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--repeats", type=int, default=7)
    a = ap.parse_args()
    torch.cuda.init()
    name, limit = card()
    T, E = a.steps, a.members
    lines = []
    for stack in a.stacks.split(","):
        for n in (int(c) for c in a.cells.split(",")):
            m, env, members = case(stack, n, T, E)
            ip = sb.InterpolationParameter()
            m.run_ensemble(ip, members)                       # warm-up: the member region, plans, kriging operators, pooled buffers
            member_loop(m, env, members[:2], ip)              # warm-up of the single path
            tb, tl, equal = [], [], True
            for _ in range(a.repeats):                        # alternating, so that both see the same state of the shared host
                t, (q, _) = timed(lambda: m.run_ensemble(ip, members))
                tb.append(t)
                t, wq = timed(lambda: member_loop(m, env, members, ip))
                tl.append(t)
                equal = equal and bool(np.array_equal(q, wq))
            t_batch, t_loop = float(np.median(tb)), float(np.median(tl))
            cs = float(n) * T * E
            line = dict(workload="forcing_ensemble", stack=stack, cells=n, steps=T, members=E, stations=64, temperature="btk",
                        precipitation="idw", repeats=a.repeats, batch_seconds=t_batch, batch_seconds_min_max=[min(tb), max(tb)],
                        loop_seconds=t_loop, loop_seconds_min_max=[min(tl), max(tl)], batch_G_cell_steps_per_s=cs / t_batch / 1e9,
                        loop_G_cell_steps_per_s=cs / t_loop / 1e9, speedup=t_loop / t_batch, batch_equals_loop=equal, card=name, power_limit=limit)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del m
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
