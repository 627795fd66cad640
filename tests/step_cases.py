"""Host rules of the step-kernel launcher (shyft_b200/csrc/sb2_capi.cu: launch_step_chunk, launch_step_range, goal_batch) restated,
the per-stack facts the step-path tests need, and the exact-sum bound the catchment sums are held to.

The rules are mirrored so that a test can state which path a case takes next to the case; the CUDA profiler's record of the launched
kernels (names and grids) then shows that the library took it."""
import math

import numpy as np

from fixtures import HBV_DEFAULT, PTGSK_DEFAULT, PTHPSK_DEFAULT, PTHSK_DEFAULT, PTSSK_DEFAULT

WARP = 32                      # cells per step group: one-warp blocks of every step kernel (SB2_BLOCK, SB2_BLOCK_B, SB2_BLOCK_C)
SPLIT_BELOW = 16000            # use_time_split: time slices while step groups x members < 16 000
RUN_CELLS_CAP = 4096           # launch_step_range: at most 4 096 steps per launch ...
CHUNK_ROUND = 128              # ... in equal chunks rounded up to a multiple of 128 steps
MAX_MEMBERS = 65535            # goal_batch: grid layers per pass
U = 2.0 ** -53                 # unit round-off of binary64

STACKS = ("pt_gs_k", "pt_hs_k", "hbv_stack", "pt_ss_k", "pt_hps_k")
STACK_ID = dict(pt_gs_k=0, pt_hs_k=1, hbv_stack=2, pt_ss_k=3, pt_hps_k=4)
UNIT_STEPS = dict(pt_gs_k=128, pt_hs_k=64, hbv_stack=64, pt_ss_k=64, pt_hps_k=64)   # SB2_UNIT_STEPS / SB2_HBV_UNIT_STEPS
MODEL = dict(pt_gs_k="PTGSKModel", pt_hs_k="PTHSKModel", hbv_stack="HbvStackModel", pt_ss_k="PTSSKModel", pt_hps_k="PTHPSKModel")
DEFAULT = dict(pt_gs_k=PTGSK_DEFAULT, pt_hs_k=PTHSK_DEFAULT, hbv_stack=HBV_DEFAULT, pt_ss_k=PTSSK_DEFAULT, pt_hps_k=PTHPSK_DEFAULT)
RESPONSES = ("avg_discharge", "charge_m3s", "snow_sca", "snow_swe", "snow_outflow", "glacier_melt", "ae_output", "pe_output")


def responses(stack):
    return RESPONSES + (("soil_outflow",) if stack == "hbv_stack" else ())


def collect_bit(name):
    """the collector-mode bit a response series is written under (wants_response)"""
    if name in ("avg_discharge", "charge_m3s"):
        return 1
    return 2 if name in ("snow_sca", "snow_swe") else 4


# parameters a catchment override changes, by index in parameter::get order: the Kirchner constants (hbv_stack: the tank), the
# snow routine's threshold temperature and the precipitation correction
OVERRIDE = dict(pt_gs_k={0: -2.9, 1: 0.9, 2: -0.13, 4: 0.8, 16: 1.2},
                pt_hs_k={0: -2.9, 1: 0.9, 2: -0.13, 5: 0.8, 10: 1.2},
                hbv_stack={3: 15.0, 4: 0.6, 5: 0.2, 7: 0.04, 9: 0.8, 13: 1.2},
                pt_ss_k={0: -2.9, 1: 0.9, 2: -0.13, 8: 0.8, 12: 1.2},
                pt_hps_k={0: -2.9, 1: 0.9, 2: -0.13, 5: 0.8, 17: 1.2})


def overridden(stack):
    p = DEFAULT[stack].copy()
    for i, v in OVERRIDE[stack].items():
        p[i] = v
    return p


def step_kernels(stack, collect, table, members=False):
    """plain names of the step kernels launch_step_chunk picks: `table` = the parameter-table (<..., false>) instantiations"""
    u = "false" if table else "true"
    if stack == "pt_gs_k":
        return [f"ptgsk_forcing_terms_kernel<{u}>", f"ptgsk_snow_kernel<{collect & 14},{u}>", f"ptgsk_response_kernel<{collect & 13},{u}>"]
    if stack == "pt_ss_k":
        return ["ptssk_run_kernel"]
    if stack == "pt_hps_k":
        return ["pthpsk_run_kernel<true>" if members else "pthpsk_run_kernel<false>"]
    return [f"hbv_run_kernel<{'true' if stack == 'hbv_stack' else 'false'},{u}>"]


def ceil_div(a, b):
    return -(-a // b)


def step_groups(n_cells):
    return ceil_div(n_cells, WARP)


def time_split(n_cells, members=1):
    return step_groups(n_cells) * members < SPLIT_BELOW


def step_grid_x(stack, n_cells, chunk, members=1):
    """grid.x of the snow / response (pt_gs_k) or run kernel for one chunk: groups x slices when split, groups when not"""
    g = step_groups(n_cells)
    return g * ceil_div(chunk, UNIT_STEPS[stack]) if time_split(n_cells, members) else g


def run_cells_chunks(n_steps, partial_steps=RUN_CELLS_CAP):
    """launch_step_range: chunk lengths of a run_cells range"""
    k = max(1, ceil_div(n_steps, partial_steps))
    even = min(partial_steps, ceil_div(ceil_div(n_steps, k), CHUNK_ROUND) * CHUNK_ROUND)
    return [min(even, n_steps - d) for d in range(0, n_steps, even)]


def ptgsk_batch_steps(n_cells, n_steps, members):
    """goal_batch for pt_gs_k: steps per chunk from the phase-pipeline scratch (five [E][ps][n] arrays within ~4 GB), when the per-slot
    partial sums (~1 GB) do not bind first"""
    E = min(members, MAX_MEMBERS)
    return max(1, min(n_steps, max(8, (4 << 30) // (E * n_cells * 40))))


def gamma(k):
    """gamma_k = k u / (1 - k u): any order of summing k + 1 doubles is within gamma_k * sum|x| of the exact sum (Higham, ASNA 4.2)"""
    return k * U / (1.0 - k * U)


def sum_error_ratios(got, X):
    """got [T] against the rows of X [T][m]: |got - sum(row)| exactly (math.fsum of got and -row is the correctly rounded error) over
    gamma(m - 1) * sum|row|, per row; an exact sum -> 0, an error over a zero bound -> inf, NaN stays NaN.  <= 1 for every
    summation order of the m values."""
    got, X = np.asarray(got, dtype=np.float64).reshape(-1), np.asarray(X, dtype=np.float64)
    err = np.array([abs(math.fsum(r)) for r in np.concatenate([got[:, None], -X], axis=1).tolist()])
    mag = np.array([math.fsum(r) for r in np.abs(X).tolist()])
    bound = gamma(X.shape[1] - 1) * mag * (1.0 + 4 * U)   # 4 u: the bound's own rounding
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(err == 0.0, 0.0, err / bound)


def worst_catchment_sum_ratio(got, series, cix, catchments=None):
    """worst sum_error_ratios of the catchment sums got [T][K] over the per-cell series [T][n] of the cells with cix == k (NaN if any)"""
    ks = range(got.shape[1]) if catchments is None else catchments
    return float(np.max([np.max(sum_error_ratios(got[:, k], series[:, cix == k])) for k in ks]))
