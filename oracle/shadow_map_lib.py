"""ctypes binding of the CPU port of the "Shadow Map Pass" (oracle/oracle_shadow_map.cpp -> oracle/_build/libvhr_shadow_map_oracle.so).
TEST INFRASTRUCTURE ONLY: the specification the CUDA pass (vhr_shadow_map_pass) is held bit-identical to.

The port is a library of its own, next to libvhr_oracle.so, built with the same compiler flags (no contraction, no fast math) when it
is missing or older than its sources.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from vulkanhybridrenderer_b200 import types as T

_ORACLE_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_ORACLE_DIR, "_build", "libvhr_shadow_map_oracle.so")
_SRCS = [os.path.join(_ORACLE_DIR, s) for s in ("oracle_shadow_map.cpp", "oracle_common.h", "shadow_map_lib.py")]
_CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wno-unknown-pragmas"]


def build(force=False):
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in _SRCS):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = f"{_SO}.{os.getpid()}.tmp"        # concurrent builders each write their own file; the rename is atomic
        subprocess.run(["g++"] + _CXXFLAGS + ["-shared", "-o", tmp, _SRCS[0]], check=True, capture_output=True)
        os.replace(tmp, _SO)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp = C.c_void_p
        L.vo_shadow_map.restype = C.c_int
        L.vo_shadow_map.argtypes = [vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_int, C.c_int, vp]
        _lib = L
    return _lib


def shadow_map(scene, pfd, W, H):
    """The "Shadow Map Pass" (vo_shadow_map): [H, W] float32 depth map of `scene` (vertices / indices / primitives) seen from
    pfd's directional_light.projview. Raises ValueError for a projview the pass rejects."""
    v = np.ascontiguousarray(scene.vertices); i = np.ascontiguousarray(scene.indices, np.uint32); p = np.ascontiguousarray(scene.primitives)
    assert v.dtype == T.Vertex and p.dtype == T.Primitive
    out = np.empty((H, W), np.float32)
    pfd = np.ascontiguousarray(pfd)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    if lib().vo_shadow_map(ptr(v), len(v), ptr(i), len(i), ptr(p), len(p), ptr(pfd), int(W), int(H), ptr(out)) != 0:
        raise ValueError("directional_light.projview is not finite or not affine (last row neither (0, 0, 0, 1) nor zero)")
    return out
