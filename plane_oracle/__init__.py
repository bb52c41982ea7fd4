"""ctypes loader of plane_oracle/libgpd_plane_oracle.so — the CPU restatement of the support-plane fit of
`sample_above_plane` (include/gpd_b200_plane.h).

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/plane_bench.py. Nothing under gpd_b200/ imports this package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from gpd_b200 import abi
from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgpd_plane_oracle.so")
_LIB = None


def build(force=False):
    src = os.path.join(_HERE, "plane_oracle.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"], env={**os.environ, "CXX": "g++"})
    return _SO


def lib():
    global _LIB
    if _LIB is None:
        oracle.lib()  # libgpd_oracle.so (pcl::eigen33) is loaded first
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        vp = C.c_void_p
        L.gpdo_sample_above_plane.argtypes = [vp, C.c_int32, C.POINTER(abi.PlaneParams), vp, C.POINTER(abi.PlaneInfo), vp,
                                              C.c_int32]
        _LIB = L
    return _LIB


def sample_above_plane(xyz, pp=None, nthreads=0):
    """Cloud::sampleAbovePlane as specified by include/gpd_b200_plane.h: (off-plane indices ascending, info dict with
    `counts` = inlier count per hypothesis, -1 where the triple is invalid). Empty indices = the plane fit failed."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
    if pp is None:
        pp = abi.default_plane_params()
    idx = np.zeros(max(len(xyz), 1), np.int32)
    counts = np.zeros(pp.num_hypotheses, np.int32)
    info = abi.PlaneInfo()
    n = lib().gpdo_sample_above_plane(xyz.ctypes.data_as(C.c_void_p), len(xyz), C.byref(pp), idx.ctypes.data_as(C.c_void_p),
                                      C.byref(info), counts.ctypes.data_as(C.c_void_p), nthreads or oracle.num_threads())
    if n < 0:
        raise RuntimeError(f"gpdo_sample_above_plane failed: {n}")
    out = abi.plane_info_to_dict(info)
    out["counts"] = counts
    return idx[:n].copy(), out
