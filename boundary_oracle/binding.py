"""ctypes binding of boundary_oracle/libfe_boundary_oracle.so: the CPU oracle's tolerance-boundary report over all
ten kinds of include/fe_b200.h (fe_enable_boundary_report_all).

TEST INFRASTRUCTURE ONLY, like oracle/oracle_binding.py, whose Params and point conventions it takes.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import oracle_binding as ob

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

KINDS = 10
KIND_NAMES = ("ring clustering", "cross-ring merge", "3DSC support", "3DSC density", "crop box", "ring windows",
              "diameter gate", "3DSC shells", "3DSC elevation", "3DSC azimuth")


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libfe_boundary_oracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
    return _LIB


def process_batch_boundary_all(params, points, scan_offsets, roll_pitch, eps_m=1e-6, mode=1, n_threads=1):
    """(B, 10) int64 counts of kinds 0-9 within eps_m; columns 0-3 are ob.process_batch_boundary's."""
    c = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
    offs = np.ascontiguousarray(scan_offsets, np.int64)
    rp = np.ascontiguousarray(roll_pitch, np.float64).reshape(-1)
    B = len(offs) - 1
    out = np.zeros((max(B, 1), KINDS), np.int64)
    p = C.c_void_p
    st = lib().feo_process_batch_boundary_all(C.byref(params), c.ctypes.data_as(p), offs.ctypes.data_as(p),
                                              rp.ctypes.data_as(p), C.c_int32(B), C.c_int32(mode), C.c_int32(n_threads),
                                              C.c_double(eps_m), out.ctypes.data_as(p))
    assert st == 0, st
    return out[:B]


