"""Register and stack budgets of the kernels a calibration batch with a routed-discharge target runs (cuobjdump on the cross-compiled
library, no GPU needed): the member-capable step kernels, which write each member's cell discharge at its own offset, and the routing
kernels with their member dimension.  The numbers are those of the build that introduced the per-member offsets (the step kernels' were
unchanged by it, except ptgsk_response_kernel<1, false>: 124 -> 126 registers); a change beyond them is a change of the batch's occupancy."""
import re
import shutil
import subprocess

import pytest

# exact mangled name -> (max registers per thread, max bytes of stack)
BUDGET = {
    "_ZN3sb221ptgsk_response_kernelILi1ELb0EEEvNS_12PtgskRunArgsE": (126, 0),    # the batch's pt_gs_k response kernel with a routed target
    "_ZN3sb221ptgsk_response_kernelILi5ELb0EEEvNS_12PtgskRunArgsE": (126, 0),
    "_ZN3sb221ptgsk_response_kernelILi9ELb0EEEvNS_12PtgskRunArgsE": (124, 0),
    "_ZN3sb221ptgsk_response_kernelILi13ELb0EEEvNS_12PtgskRunArgsE": (126, 0),
    "_ZN3sb214hbv_run_kernelILb0ELb0EEEvNS_10HbvRunArgsE": (128, 80),             # pt_hs_k with overrides / batch
    "_ZN3sb214hbv_run_kernelILb1ELb0EEEvNS_10HbvRunArgsE": (96, 56),              # hbv_stack with overrides / batch
    "_ZN3sb217pthpsk_run_kernelILb1EEEvNS_10HpsRunArgsE": (128, 192),             # pt_hps_k batch
    "_ZN3sb225route_local_inflow_kernelEPKdlllllPKiS3_S3_S3_S1_iiPdlll": (32, 0),
    "_ZN3sb224route_river_level_kernelEPKiS1_S1_S1_S1_PKdilS3_PdS4_l": (32, 0),
    "_ZN3sb220route_history_kernelEPKdPdlll": (32, 0),
}


def test_routed_batch_kernels_keep_their_register_budgets():
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
            found[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    for kernel, (max_reg, max_stack) in BUDGET.items():
        assert kernel in found, f"{kernel}: kernel not found in the library"
        reg, stack = found[kernel]
        assert reg <= max_reg, f"{kernel}: {reg} registers, budget {max_reg}"
        assert stack <= max_stack, f"{kernel}: {stack} B of stack (spills), budget {max_stack}"
