"""The host-rule mirrors and the exact-sum bound of tests/step_cases.py, which tests/test_gpu_step_paths.py relies on, checked without a
device: the launcher's numbers the GPU cases quote, and a bound that admits every summation order but not a missing term."""
import math

import numpy as np

import step_cases as sc


def test_time_split_threshold():
    assert sc.step_groups(512017) == 16001 and not sc.time_split(512017)
    assert sc.step_groups(511968) == 15999 and sc.time_split(511968)
    assert not sc.time_split(512000) and not sc.time_split(240, 2000) and sc.time_split(240, 1999)
    assert sc.step_grid_x("pt_gs_k", 100, 129) == 4 * 2 and sc.step_grid_x("pt_hs_k", 100, 129) == 4 * 3
    assert sc.step_grid_x("pt_ss_k", 512017, 150) == 16001


def test_chunk_rules():
    assert sc.run_cells_chunks(5000) == [2560, 2440]
    assert sc.run_cells_chunks(4096) == [4096] and sc.run_cells_chunks(4097) == [2176, 1921]
    assert sc.run_cells_chunks(150) == [150] and sc.run_cells_chunks(1) == [1]
    assert sc.ptgsk_batch_steps(240, 1440, 2000) == 223     # 4 GiB / (2 000 x 240 x 40 B)
    assert sc.ptgsk_batch_steps(240, 1440, 1) == 1440
    assert sc.ptgsk_batch_steps(64, 96, 65537) == 25         # the pass holds 65 535 members


def test_kernel_names():
    assert sc.step_kernels("pt_gs_k", 15, table=False) == ["ptgsk_forcing_terms_kernel<true>", "ptgsk_snow_kernel<14,true>",
                                                           "ptgsk_response_kernel<13,true>"]
    assert sc.step_kernels("pt_gs_k", 6, table=True)[1:] == ["ptgsk_snow_kernel<6,false>", "ptgsk_response_kernel<4,false>"]
    assert sc.step_kernels("hbv_stack", 1, table=True) == ["hbv_run_kernel<true,false>"]
    assert sc.step_kernels("pt_hps_k", 1, table=False) == ["pthpsk_run_kernel<false>"]


def test_sum_bound_admits_every_order_and_no_missing_term():
    rng = np.random.default_rng(3)
    for m in (1, 2, 7, 160, 1000):
        X = rng.standard_normal((40, m)) * np.exp(rng.uniform(-20, 20, (40, m)))   # signed, wide range: charges
        for order in (X, X[:, ::-1], np.sort(X, axis=1), X[:, rng.permutation(m)]):
            naive = np.array([sum(row) for row in order.tolist()])                   # left to right in binary64
            assert np.all(sc.sum_error_ratios(naive, X) <= 1.0)
        pairwise = X.sum(axis=1)                                                      # numpy's pairwise order
        assert np.all(sc.sum_error_ratios(pairwise, X) <= 1.0)
        rounded = np.array([math.fsum(row) for row in X.tolist()])                  # the correctly rounded sum
        assert np.all(sc.sum_error_ratios(rounded, X) <= 1.0)
        if m > 1:
            Q = rng.uniform(0.5, 1.5, (40, m))                                        # discharges of one size
            short = np.array([sum(row[:-1]) for row in Q.tolist()])                   # the last slot skipped
            assert np.all(sc.sum_error_ratios(short, Q) > 1.0)
    assert sc.gamma(0) == 0.0
    assert sc.sum_error_ratios([1.0 + 2 ** -52], [[1.0]])[0] == math.inf   # one cell: the sum must be the value itself
    assert np.isnan(sc.sum_error_ratios([1.0], [[np.nan, 1.0]])[0])
