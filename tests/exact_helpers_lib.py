"""ctypes binding of the device test harness of vhr_common.cuh's exactly-rounded helpers (tests/csrc/exact_helpers_harness.cu ->
tests/csrc/_build/libvhr_exact_helpers.so).

The harness includes the library's header and is compiled with the library's nvcc flags, so the helpers it runs are the ones the kernels
run. It is built where nvcc is (sm_100a cross-compiles without a GPU) when it is missing or older than its sources, and travels with the
tree like libvhr_b200.so. Every entry point takes device pointers (torch tensors) and enqueues on the default stream.
"""
import ctypes as C
import os
import subprocess

from vulkanhybridrenderer_b200 import build as B

_TESTS_DIR = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_TESTS_DIR)
SRC = os.path.join(_TESTS_DIR, "csrc", "exact_helpers_harness.cu")
HEADER = os.path.join(_ROOT, "vulkanhybridrenderer_b200", "csrc", "vhr_common.cuh")
SO = os.path.join(_TESTS_DIR, "csrc", "_build", "libvhr_exact_helpers.so")

REPORT_RECORDS = 64


def build(force=False):
    if force or not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in (SRC, HEADER)):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        tmp = f"{SO}.{os.getpid()}.tmp"        # concurrent builders each write their own file; the rename is atomic
        r = subprocess.run([B.NVCC] + B.NVCC_FLAGS + ["-shared", "-o", tmp, SRC], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"building {SO} failed:\n{r.stdout}{r.stderr}")
        os.replace(tmp, SO)
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, i = C.c_void_p, C.c_int
        for name, args in (("eh_sqrt_sweep", [vp]), ("eh_sqrt_eval", [vp, vp, vp, i]), ("eh_div_eval", [vp, vp, i, vp, vp, vp, vp, vp]),
                           ("eh_div_sweep", [vp, i, vp, i, i, vp]), ("eh_bilinear_sweep", [i, vp]), ("eh_bilinear_eval", [vp, i, i, vp, vp, vp]),
                           ("eh_wrap_sweep", [i, vp]), ("eh_sincos_eval", [vp, i, vp, vp]), ("eh_report_size", [])):
            getattr(L, name).argtypes = args
            getattr(L, name).restype = C.c_int
        assert L.eh_report_size() == 16 + REPORT_RECORDS * 16
        _lib = L
    return _lib


def call(name, *args):
    """Calls an entry point; torch tensors are passed as device pointers. Raises on a launch error."""
    import torch
    conv = [C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args]
    rc = getattr(lib(), name)(*conv)
    if rc != 0:
        raise RuntimeError(f"{name}: CUDA error {rc}")


def new_report():
    import torch
    return torch.zeros(2 + REPORT_RECORDS * 2, dtype=torch.int64, device="cuda")


def read_report(rep):
    """(mismatches, checked, [up to 64 records of four uint32 words])."""
    import torch
    torch.cuda.synchronize()
    h = rep.cpu().numpy()
    n, checked = int(h[0]), int(h[1])
    recs = h[2:].view("<u4").reshape(REPORT_RECORDS, 4)[: min(n, REPORT_RECORDS)]
    return n, checked, [tuple(int(x) for x in r) for r in recs]
