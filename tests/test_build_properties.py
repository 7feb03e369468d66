"""Compile-time properties the measured numbers depend on, read from the built library (no GPU needed): the kernels are
compiled for sm_100a and keep the register budgets their occupancy was tuned for (DESIGN.md section 2: primary and
early-bounce trace 64 registers = 4 blocks of 256 threads per SM, late-bounce trace 80 = 3 blocks, shade 64, miss 32),
and the path has no tensor-core / TMA instructions (no stage is a contraction: BASELINE.json north_star)."""
import os
import re
import shutil
import subprocess

import pytest

from helpers import LIB

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB),
                                reason="needs the built library and cuobjdump")

# mangled-name fragment -> (max registers per thread, max bytes of stack = spills + local arrays); every kernel whose
# mangled name contains the fragment is held to it
BUDGET = {
    # the stage kernels
    "rt_trace_kernelILb1ELi4E": (64, 64),
    "rt_trace_kernelILb0ELi4E": (64, 64),
    "rt_trace_kernelILb0ELi3E": (80, 16),
    "15rt_shade_kernel11": (64, 96),
    "14rt_miss_kernel11": (32, 32),
    # the ray queries (csrc/rt_query.cu): the wide bounce trace's 64 registers (4 blocks of 256 threads per SM) and no
    # more stack than it has (24 bytes: the leaf and accept counters, spilled once per leaf, outside the node step and
    # the triangle loop)
    "rt_query_kernelILb0E": (64, 24),       # closest hit
    "rt_query_kernelILb1E": (64, 24),       # occlusion
    # first-surface AOVs, from -Xptxas -v
    "rt_aov_surface_kernel": (32, 0),
    "rt_aov_accumulate_kernel": (64, 16),
    # cast_rays, from -Xptxas -v
    "rt_cast_rays_raygen_kernel": (24, 0),
    "rt_cast_rays_accumulate_kernel": (32, 0),
    # masked sample passes, from -Xptxas -v
    "rt_trace_kernelILb1ELi4ELb1E": (64, 24),       # the masked primary trace: the unmasked one's 64 registers and
                                                    # 24-byte frame
    "rt_accumulate_masked_kernel": (40, 0),
    "rt_resolve_counts_kernel": (32, 0),
    # many views, from -Xptxas -v
    "rt_trace_kernelILb1ELi4ELb0ELb1E": (64, 24),   # the unmasked primary trace's 64 registers and 24-byte frame
    # sky tiles: 64 registers (4 blocks of 256 threads per SM) and no spills
    "13rt_sky_kernel": (64, 16),                     # exact
    "18rt_sky_kernel_fast": (64, 16),                # fast
}


def test_stage_kernels_keep_their_register_budgets():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True).stdout
    kernels = [(m.group(1), int(m.group(2)), int(m.group(3)))
               for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)]
    missing = [key for key in BUDGET if not any(key in name for name, _, _ in kernels)]
    assert not missing, f"kernels missing from the library: {missing}"
    over = [f"{name}: {regs} registers, {stack} bytes of stack (budget {BUDGET[key][0]}, {BUDGET[key][1]})"
            for key in BUDGET for name, regs, stack in kernels
            if key in name and (regs > BUDGET[key][0] or stack > BUDGET[key][1])]
    assert not over, "over budget (occupancy would drop, or spills in the hot loops):\n" + "\n".join(over)


def test_library_is_sm_100a_without_tensor_or_tma_instructions():
    elfs = subprocess.run(["cuobjdump", "-lelf", LIB], capture_output=True, text=True).stdout
    assert "sm_100a" in elfs and "sm_90" not in elfs
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    assert len(sass) > 100000
    assert not re.search(r"UTMALDG|UTCMMA|UTCHMMA|LDTM|HMMA|WGMMA", sass)
