"""Register and stack budget of the kernel a forcing-ensemble run adds (cuobjdump on the cross-compiled library, no GPU needed): the
scatter of each member's interpolated window and of the parent's state into the internal member region.  The numbers are those of the
build that introduced it."""
import re
import shutil
import subprocess

import pytest

# exact mangled name -> (max registers per thread, max bytes of stack)
BUDGET = {
    "_ZN3sb223ensemble_scatter_kernelEPKdllllPdll": (30, 0),
}


def test_ensemble_kernels_keep_their_register_budgets():
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
