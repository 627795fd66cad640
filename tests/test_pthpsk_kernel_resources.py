"""Build-time guard of the two pt_hps_k step kernels (cuobjdump on the cross-compiled library, no GPU needed): the run_cells
instantiation keeps its registers and stack, and the calibration-batch instantiation stays at the same launch bound with at most
a few member offsets more on the stack."""
import re
import shutil
import subprocess

import pytest

# kernel name fragment -> (max registers per thread, max bytes of stack), with sm_100a and the library's nvcc flags
BUDGET = {
    "pthpsk_run_kernelILb0E": (128, 184),   # run_cells: 16 resident warps (launch bound (128, 4)); 184 B as before the batch existed
    "pthpsk_run_kernelILb1E": (128, 248),   # calibration batch: measured 128 / 192, allowed up to 64 B over the run_cells kernel
}


def test_pthpsk_kernels_keep_their_register_budgets():
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
        assert stack <= max_stack, f"{frag}: {stack} B of stack, budget {max_stack}"
