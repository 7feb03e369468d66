"""Compile-time budget of the ray-query kernels (csrc/rt_query.cu), read from the built library (no GPU needed): both
instantiations keep the 64 registers of 4 blocks of 256 threads per SM they are built for (the wide bounce trace's
budget), with no more stack than that kernel (24 bytes: the leaf and accept counters, spilled once per leaf, outside the
node step and the triangle loop)."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing_c_b200", "csrc", "libraytracer_gpu.so")

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB),
                                reason="needs the built library and cuobjdump")

BUDGET = {   # mangled-name fragment -> (max registers per thread, max bytes of stack)
    "rt_query_kernelILb0E": (64, 24),       # closest hit
    "rt_query_kernelILb1E": (64, 24),       # occlusion
}


def test_query_kernels_keep_their_register_budget():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
    found = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        for key in BUDGET:
            if key in m.group(1):
                found[key] = (int(m.group(2)), int(m.group(3)))
    assert set(found) == set(BUDGET), f"kernels missing from the library: {set(BUDGET) - set(found)}"
    for key, (regs, stack) in found.items():
        assert regs <= BUDGET[key][0], f"{key}: {regs} registers (budget {BUDGET[key][0]}) — occupancy would drop"
        assert stack <= BUDGET[key][1], f"{key}: {stack} bytes of stack (budget {BUDGET[key][1]}) — spills in the walk"
