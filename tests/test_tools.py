"""The measurement tools start without a GPU: each parses its command line with the shared module (tools/benchkit.py)
and all its imports in place."""
import os
import subprocess
import sys

import pytest

from helpers import ROOT

TOOLS = ["adaptive_bench", "aov_bench", "cast_rays_bench", "query_bench", "refit_bench", "views_bench",
         "profile_render", "config_sweep"]


@pytest.mark.parametrize("tool", TOOLS)
def test_tool_help(tool):
    run = subprocess.run([sys.executable, os.path.join(ROOT, "tools", f"{tool}.py"), "--help"],
                         capture_output=True, text=True, timeout=300)
    assert run.returncode == 0, run.stderr
    assert run.stdout.startswith("usage:")
