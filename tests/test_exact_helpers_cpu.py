"""The device harness of vhr_common.cuh's exact helpers builds for sm_100a and runs the library's own header (no copy of the helpers)."""
import os
import re
import subprocess

import pytest

import exact_helpers_lib as E
from vulkanhybridrenderer_b200 import build as B


def test_harness_cross_compiles_for_sm_100a_from_the_real_header(tmp_path):
    if not os.path.exists(B.NVCC):
        pytest.skip(f"no nvcc at {B.NVCC}")
    so = str(tmp_path / "h.so")
    subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-shared", "-o", so, E.SRC], check=True, capture_output=True)
    elf = subprocess.run([os.path.join(os.path.dirname(B.NVCC), "cuobjdump"), "-lelf", so], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in elf, elf
    deps = subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-M", E.SRC], check=True, capture_output=True, text=True).stdout
    assert os.path.realpath(E.HEADER) in {os.path.realpath(d) for d in deps.replace("\\\n", " ").split() if d.endswith(".cuh")}, deps
    src = open(E.SRC).read()
    for helper in ("exact_divisor", "div_exact", "div_exact_flag", "div_exact_flag_bounded", "sqrt_exact", "bilinear_setup", "subtexel_rn",
                   "wrap_repeat", "wrap_texel"):
        assert not re.search(rf"\b(int|float|void|ExactDivisor)\s+{helper}\s*\(", src), f"the harness redefines {helper}"
