"""The G-buffer kernel's two instances (single-GPU and partitioned) cross-compile for sm_100a with the library's flags, within the
128-thread launch bounds and without spilling registers."""
import os
import re
import subprocess

import pytest

from vulkanhybridrenderer_b200 import build as B


def test_gbuffer_kernel_instances_compile_without_spills(tmp_path):
    if not os.path.exists(B.NVCC):
        pytest.skip(f"no nvcc at {B.NVCC}")
    src = os.path.join(B.CSRC, "trace_kernels.cu")
    r = subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "t.o")], check=True, capture_output=True, text=True)
    log = r.stdout + r.stderr
    found = {}
    for m in re.finditer(r"Compiling entry function '\S*gbuffer_kernelILb([01])E\S*' for 'sm_100a'\n(.*?Used \d+ registers[^\n]*)", log, re.S):
        found[m.group(1)] = m.group(2)
    assert set(found) == {"0", "1"}, log[-3000:]
    for inst, info in found.items():
        assert "0 bytes spill stores, 0 bytes spill loads" in info, (inst, info)
        regs = int(re.search(r"Used (\d+) registers", info).group(1))
        assert regs <= 65536 // 128 // 2, (inst, info)          # at least two 128-thread blocks per SM
