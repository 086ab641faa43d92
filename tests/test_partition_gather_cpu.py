"""The composition kernels' instances cross-compile for sm_100a with the library's flags, without spilling registers: the 27 mode
combinations of composition_kernel and present_kernel, each as the single-GPU instance (<false>) and as the instance that also stores
every texel into the output rank's render output (<true>, VHR_OPT_OUTPUT_RANK). A <true> instance keeps as many resident 256-thread
blocks per SM as its <false> instance."""
import os
import re
import subprocess

import pytest

from vulkanhybridrenderer_b200 import build as B

MODES = [(s, a, r) for s in range(3) for a in range(3) for r in range(3)]


def _blocks_per_sm(regs):
    """resident 256-thread blocks per SM of sm_100a for `regs` registers per thread: 64 K registers, allocated per warp in units of
    256 (8 per thread), at most 2048 threads"""
    per_thread = (regs + 7) // 8 * 8
    return min(2048 // 256, 65536 // (per_thread * 256))


def test_composition_instances_compile_without_spills(tmp_path):
    if not os.path.exists(B.NVCC):
        pytest.skip(f"no nvcc at {B.NVCC}")
    src = os.path.join(B.CSRC, "composition_kernels.cu")
    r = subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "c.o")], check=True, capture_output=True, text=True)
    log = r.stdout + r.stderr
    found = {}
    for m in re.finditer(r"Compiling entry function '_ZN3vhr\d+((?:composition|present)_kernelI\w+?EE)\S*' for 'sm_100a'\n(.*?Used \d+ registers[^\n]*)", log, re.S):
        found[m.group(1)] = m.group(2)
    want = {f"composition_kernelILi{s}ELi{a}ELi{r}ELb{g}EE" for s, a, r in MODES for g in (0, 1)} | {"present_kernelILb0EE", "present_kernelILb1EE"}
    assert set(found) == want, (sorted(set(found) ^ want), log[-3000:])
    assert len(want) == 56
    regs = {}
    for name, info in found.items():
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in info, (name, info)
        regs[name] = int(re.search(r"Used (\d+) registers", info).group(1))
    pairs = [(f"composition_kernelILi{s}ELi{a}ELi{r}ELb0EE", f"composition_kernelILi{s}ELi{a}ELi{r}ELb1EE") for s, a, r in MODES]
    for single, gather in pairs + [("present_kernelILb0EE", "present_kernelILb1EE")]:
        assert _blocks_per_sm(regs[gather]) >= _blocks_per_sm(regs[single]), (single, regs[single], gather, regs[gather])
