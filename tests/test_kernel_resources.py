"""Build-time guard of the hot kernels' register budgets (cuobjdump on the cross-compiled library, no GPU needed): every one of these
numbers is a measured optimum (profiles/README.md) and a silent change of it -- a new launch bound, a few more live values -- costs
several per cent on the B200 before any test notices."""
import re
import shutil
import subprocess

import pytest

# kernel name fragment -> (max registers per thread, max bytes of stack = spills)
BUDGET = {
    "ptgsk_forcing_terms_kernel": (72, 0),          # 28 resident warps; 94 registers (launch bound (128, 1)) cost 2.4 ms per year
    "ptgsk_snow_kernelILi0E": (128, 256),           # 16 one-warp blocks per SM
    "ptgsk_response_kernelILi1E": (122, 0),         # 16 one-warp blocks per SM, no spills
    "hbv_run_kernelILb0E": (128, 64),               # pt_hs_k: 16 resident warps
    "hbv_run_kernelILb1E": (96, 160),               # hbv_stack: 20 resident warps
    "pthpsk_run_kernelILb0E": (128, 184),           # pt_hps_k run_cells: 16 resident warps (launch bound (128, 4)); 184 B as before the batch existed
    "pthpsk_run_kernelILb1E": (128, 248),           # pt_hps_k calibration batch: measured 128 / 192, allowed up to 64 B over the run_cells kernel
    "dense_apply_dmma_kernelILi6ELi2ELi0ELb1ELi16ELi32E": (80, 0),   # compacted IDW, 10 neighbours
    "dense_apply_dmma_kernelILi16ELi2ELi1ELb0ELi16ELi0E": (128, 0),  # Bayesian kriging, 64 stations
}


def test_hot_kernels_keep_their_register_budgets():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    from shyft_b200 import capi
    capi.lib()
    out = subprocess.run([cuobjdump, "--dump-resource-usage", capi.library_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump not available")
    found = {}
    name = None
    for line in out.stdout.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", line)
        if m and name:
            for frag in BUDGET:
                if frag in name:
                    found[frag] = (int(m.group(1)), int(m.group(2)))
            name = None
    for frag, (max_reg, max_stack) in BUDGET.items():
        assert frag in found, f"{frag}: kernel not found in the library"
        reg, stack = found[frag]
        assert reg <= max_reg, f"{frag}: {reg} registers, budget {max_reg}"
        assert stack <= max_stack, f"{frag}: {stack} B of stack (spills), budget {max_stack}"
