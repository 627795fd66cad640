"""The forcing-ensemble host rules of tests/ensemble_cases.py, which tests/test_gpu_ensemble.py relies on, checked without a device:
padding to the warp, internal catchment numbering, the slot layout of each member copy (the ground of the bit-identity argument in
DESIGN.md section 3.7) and the members per pass."""
import numpy as np

import ensemble_cases as ec


def test_padding_and_catchments_per_member():
    assert ec.layout("pt_hs_k", 203, 3, 720, 720, 4096, 6)["np"] == 224
    assert ec.layout("pt_hs_k", 203, 3, 720, 720, 4096, 6)["kp"] == 4      # the padding cells' catchment
    assert ec.layout("pt_hs_k", 224, 3, 720, 720, 4096, 6)["kp"] == 3      # a whole number of warps: no padding
    assert ec.layout("pt_hs_k", 203, 3, 720, 300, 97, 6)["window"] == 97
    assert ec.layout("pt_hs_k", 203, 3, 720, 300, 4096, 6)["window"] == 300


def test_internal_numbering_is_first_appearance():
    rng = np.random.default_rng(3)
    for n in (1, 31, 32, 33, 203):
        ids = list(rng.integers(100, 105, n))
        cix = ec.first_appearance(ids)
        K = max(cix) + 1
        internal = ec.internal_catchments(cix, K, 5)
        assert ec.first_appearance(internal) == internal, n     # sb2_model_create numbers them e * kp + k, as build_member_region checks


def test_member_copies_have_the_parents_slots():
    rng = np.random.default_rng(5)
    for n in (1, 31, 33, 65, 203, 300):
        cix = ec.first_appearance(list(rng.integers(0, 4, n) // 2 + np.arange(n) // 40))
        K = max(cix) + 1
        E = 4
        lay = ec.layout("hbv_stack", n, K, 10, 10, 10, E)
        slot, by_cat = ec.slots(cix)
        islot, iby_cat = ec.slots(ec.internal_catchments(cix, K, E))
        per_copy = max(islot) // E + 1
        for e in range(E):
            for c in range(n):   # the same lane, the same slot number within the copy
                assert islot[e * lay["np"] + c] - e * per_copy == slot[c]
            for k in range(K):   # each real catchment sums the same slots in the same order
                assert [s - e * per_copy for s in iby_cat[e * lay["kp"] + k]] == by_cat[k]


def test_members_per_pass():
    # 100 000 cells x 240 steps: pt_gs_k 1.93 GB a member; 32 GiB less 2.2 GB of windows and partial sums holds 16, so 51 members go in 4
    # passes of 13, the last with one spare copy
    lay = ec.layout("pt_gs_k", 100000, 10, 240, 240, 4096, 51)
    assert lay["per_member"] == 8 * 100000 * (2400 + 9) + 16 * 240 * 10
    assert (lay["passes"], lay["per_pass"]) == (4, 13) and ec.pass_sizes(51, 13) == [13, 13, 13, 12]
    lay = ec.layout("hbv_stack", 100000, 10, 240, 240, 4096, 51)
    assert (lay["passes"], lay["per_pass"]) == (2, 26)
    assert ec.layout("hbv_stack", 10000, 10, 240, 240, 4096, 51)["passes"] == 1
    # the GPU case sized for two passes: 10 000 cells x 21 600 steps of pt_hs_k is 8.7 GB a member, 3 members in passes of 2 and 1
    lay = ec.layout("pt_hs_k", 10000, 3, 21600, 21600, 21600, 3)
    assert lay["per_member"] == 8 * 10016 * (5 * 21600 + 13) + 16 * 21600 * 4
    assert (lay["passes"], lay["per_pass"]) == (2, 2) and ec.pass_sizes(3, 2) == [2, 1]
    assert ec.layout("pt_hs_k", 20000, 3, 21600, 21600, 21600, 2)["per_pass"] == 1
    assert ec.layout("pt_hs_k", 20000, 3, 21600, 21600, 21600, 1)["passes"] == 1   # at least one member a pass
