"""lean::k_step_observe, the step with a face at 16 resident warps per SM: it exists for every face variant and keeps
its warps' state in registers (no stack, no spills), which is what it is for (DESIGN.md §8)."""
import os
import re
import shutil
import subprocess

import pytest


def test_lean_step_kernels_do_not_spill():
    import ddz_b200 as D
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-res-usage", D.native.LIB_PATH], capture_output=True, text=True).stdout
    found = re.findall(r"Function _ZN3ddz4lean14k_step_observeILi(\d)EE\S*:\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    assert sorted(int(v) for v, *_ in found) == [0, 1, 2, 3]
    for v, reg, stack, local in found:
        assert int(stack) == 0 and int(local) == 0, v
        assert 72 < int(reg) <= 128, v     # more than k_env's 72, within 16 warps per SM
