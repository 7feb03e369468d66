"""include/rt_fastdiv.h: the multiply-high division the primary trace uses for path id -> (pixel, sample) and
tile -> (x, y) must equal `/` for every dividend of the range it was made for (exhaustive for small ranges,
strided plus every multiple-of-d boundary for the large ones)."""
import os
import subprocess

from helpers import ROOT


def test_fastdiv_equals_division(tmp_path):
    exe = tmp_path / "fastdiv_check"
    subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "csrc", "fastdiv_check.c")], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert out.stdout.strip().endswith("ok")


def test_fma_division_by_1p055_is_the_ieee_quotient(tmp_path):
    """rt_shade.cuh div_1p055 (sRGB decode): x*r, exact residual, one correction == x / 1.055f for every float in [0.01, 4]."""
    exe = tmp_path / "div_const_check"
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-o", str(exe),
                    os.path.join(ROOT, "tests", "csrc", "div_const_check.c"), "-lm"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert out.stdout.strip().endswith("ok")


def test_texel_byte_to_float_by_fma_is_the_ieee_quotient(tmp_path):
    """rt_shade.cuh texel_channel: PRMT into the mantissa of 2^23 + one fused multiply-add == (float)b / 255.999f for all bytes."""
    exe = tmp_path / "texel_scale_check"
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-o", str(exe),
                    os.path.join(ROOT, "tests", "csrc", "texel_scale_check.c"), "-lm"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert out.stdout.strip().endswith("ok")
