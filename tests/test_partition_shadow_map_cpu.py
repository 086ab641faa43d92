"""The shadow-map kernels' instances (single-GPU and partitioned setup, tile and clip kernels) and the push kernel cross-compile for
sm_100a with the library's flags, without spilling registers. The clip kernel's stack frame holds its clipping polygons, as before.
A partitioned instance uses no more registers than its single-GPU one, so it keeps at least its occupancy; the push kernel keeps
four 256-thread blocks per SM."""
import os
import re
import subprocess

import pytest

from vulkanhybridrenderer_b200 import build as B

KERNELS = {"shadow_setup_kernelILb0E", "shadow_setup_kernelILb1E", "shadow_tile_kernelILb0E", "shadow_tile_kernelILb1E",
           "shadow_clip_kernelILb0E", "shadow_clip_kernelILb1E", "shadow_push_kernelE"}


def test_shadow_map_kernel_instances_compile_without_spills(tmp_path):
    if not os.path.exists(B.NVCC):
        pytest.skip(f"no nvcc at {B.NVCC}")
    src = os.path.join(B.CSRC, "shadow_map_kernels.cu")
    r = subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "s.o")], check=True, capture_output=True, text=True)
    log = r.stdout + r.stderr
    found = {}
    for m in re.finditer(r"Compiling entry function '_ZN3vhr\d+(shadow_\w+?kernel(?:ILb[01]E|E))\S*' for 'sm_100a'\n(.*?Used \d+ registers[^\n]*)", log, re.S):
        found[m.group(1)] = m.group(2)
    assert set(found) == KERNELS, log[-3000:]
    regs = {}
    for name, info in found.items():
        assert "0 bytes spill stores, 0 bytes spill loads" in info, (name, info)
        regs[name] = int(re.search(r"Used (\d+) registers", info).group(1))
        if "clip" not in name:
            assert "0 bytes stack frame" in info, (name, info)
    for k in ("setup", "tile", "clip"):
        assert regs[f"shadow_{k}_kernelILb1E"] <= regs[f"shadow_{k}_kernelILb0E"], regs
    assert regs["shadow_push_kernelE"] <= 65536 // (4 * 256), regs
