"""ctypes binding of match_oracle/libfe_match_oracle.so: the CPU restatement of fe_match_descriptors
(include/fe_b200.h, "descriptor matching").

TEST INFRASTRUCTURE ONLY, like oracle/oracle_binding.py: never imported by the feature_extraction_b200 package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

DESC_LEN = 1980
RECORD_FLOATS = 1996


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "libfe_match_oracle.so")
        if not os.path.exists(path):
            build()
        _LIB = C.CDLL(path)
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def match_descriptors(query, ref, query_offsets=None, ref_offsets=None, n_threads=1):
    """feo_match_descriptors on the CPU.  `query` / `ref`: (K, 1980) bins or (K, 1996) records (stride 1996, bins at
    offset 5); no offsets = one group.  -> best (n,) int64, shift (n,) int32, dist2 (n,) float32, second_dist2 (n,)"""
    def rows(a):
        a = np.ascontiguousarray(a, np.float32)
        assert a.ndim == 2 and a.shape[1] in (DESC_LEN, RECORD_FLOATS), a.shape
        first = 5 if a.shape[1] == RECORD_FLOATS else 0
        return a, a.shape[1], C.c_void_p(a.ctypes.data + 4 * first if len(a) else None)
    q, qs, qp = rows(query)
    r, rs, rp = rows(ref)
    if query_offsets is None and ref_offsets is None:
        query_offsets, ref_offsets = [0, len(q)], [0, len(r)]
    qo = np.ascontiguousarray(query_offsets, np.int64)
    ro = np.ascontiguousarray(ref_offsets, np.int64)
    G = len(qo) - 1
    n = int(qo[-1] - qo[0]) if G >= 0 else 0
    best = np.zeros(max(n, 1), np.int64)
    shift = np.zeros(max(n, 1), np.int32)
    d = np.zeros(max(n, 1), np.float32)
    sd = np.zeros(max(n, 1), np.float32)
    st = lib().feo_match_descriptors(qp, C.c_int64(qs), _p(qo), rp, C.c_int64(rs), _p(ro), C.c_int32(G), C.c_int32(n_threads),
                                     _p(best), _p(shift), _p(d), _p(sd))
    assert st == 0, st
    return best[:n], shift[:n], d[:n], sd[:n]
