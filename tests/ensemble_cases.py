"""Host rules of the forcing-ensemble run (shyft_b200/csrc/sb2_capi.cu: ensemble_layout, build_member_region, build_slots) restated, so
that a test can state the layout, the internal catchment numbering and the passes a case takes next to the case."""
import math

WARP = 32
BUDGET = 32 << 30          # kEnsembleBudget: the device buffers of one call
MAX_MEMBERS = 65535        # grid z of the scatter kernel
N_STATE = dict(pt_gs_k=9, pt_hs_k=13, hbv_stack=15, pt_ss_k=8, pt_hps_k=24)


def layout(stack, n, n_catch, T, count, window_steps, members):
    """-> dict(np, kp, window, per_member, per_pass, passes) as ensemble_layout computes them"""
    np_ = (n + WARP - 1) // WARP * WARP
    kp = n_catch + (1 if np_ > n else 0)
    W = min(window_steps, count)
    fixed = 6 * 8 * W * n + (1 << 30)   # the member window, up to five windows from the model's own sources, the partial sums
    per_member = 8 * np_ * (5 * W * (2 if stack == "pt_gs_k" else 1) + N_STATE[stack]) + 16 * T * kp
    cap = max(1, min(members, MAX_MEMBERS, max(0, BUDGET - fixed) // per_member))
    passes = math.ceil(members / cap)
    return dict(np=np_, kp=kp, window=W, per_member=per_member, per_pass=math.ceil(members / passes), passes=passes)


def pass_sizes(members, per_pass):
    """members of each pass; the region holds per_pass copies, a shorter last pass fills the spare ones with its last member"""
    return [min(per_pass, members - e0) for e0 in range(0, members, per_pass)]


def first_appearance(ids):
    """catchment index of every cell: ids numbered in order of first appearance (update_ix_to_id_mapping, sb2_model_create)"""
    ix, out = {}, []
    for c in ids:
        out.append(ix.setdefault(c, len(ix)))
    return out


def internal_catchments(cix_of_cell, n_catch, members):
    """internal catchment id of every internal cell: member e's copy of cell c is cell e * np + c with id e * kp + cix; padding kp - 1"""
    n = len(cix_of_cell)
    np_ = (n + WARP - 1) // WARP * WARP
    kp = n_catch + (1 if np_ > n else 0)
    return [e * kp + (cix_of_cell[c] if c < n else n_catch) for e in range(members) for c in range(np_)]


def slots(cix_of_cell):
    """build_slots: one slot per run of equal catchment index within a 32-cell warp -> (slot of each cell, slots of each catchment in order)"""
    slot, by_cat, ns = [], {}, 0
    for i, k in enumerate(cix_of_cell):
        if i % WARP == 0 or k != cix_of_cell[i - 1]:
            by_cat.setdefault(k, []).append(ns)
            ns += 1
        slot.append(ns - 1)
    return slot, by_cat
