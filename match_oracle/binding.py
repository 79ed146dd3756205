"""ctypes binding of match_oracle/libfe_match_oracle.so: the CPU restatements of fe_match_descriptors,
fe_register_matches, fe_odometry and fe_loop_closures (include/fe_b200.h, "descriptor matching", "registration",
"odometry", "loop closures").

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


def register_matches(query_kp, ref_kp, best, query_offsets, ref_offsets, inlier_radius=0.5, min_separation=1.0,
                     max_hypotheses=512, min_inliers=16, refine_iterations=4):
    """feo_register_matches on the CPU.  query_kp / ref_kp: (K, 4) float32 keypoints addressed by absolute row;
    best: (qo[-1] - qo[0],) int64.  -> dict of pose (G, 4) float64 {c, s, tx, ty}, rms (G,), n_inliers (G,),
    n_hypotheses (G,), status (G,) int32 and assoc (n,) int64."""
    q = np.ascontiguousarray(query_kp, np.float32).reshape(-1, 4)
    r = np.ascontiguousarray(ref_kp, np.float32).reshape(-1, 4)
    b = np.ascontiguousarray(best, np.int64).reshape(-1)
    qo = np.ascontiguousarray(query_offsets, np.int64)
    ro = np.ascontiguousarray(ref_offsets, np.int64)
    G = len(qo) - 1
    n = int(qo[-1] - qo[0])
    assert len(b) == n, (len(b), n)
    out = {"pose": np.zeros((max(G, 1), 4)), "rms": np.zeros(max(G, 1)), "n_inliers": np.zeros(max(G, 1), np.int32),
           "n_hypotheses": np.zeros(max(G, 1), np.int32), "status": np.zeros(max(G, 1), np.int32),
           "assoc": np.zeros(max(n, 1), np.int64)}
    st = lib().feo_register_matches(
        _p(q) if len(q) else None, _p(r) if len(r) else None, _p(b) if n else None, _p(qo), _p(ro), C.c_int32(G),
        C.c_double(inlier_radius), C.c_double(min_separation), C.c_int32(max_hypotheses), C.c_int32(min_inliers),
        C.c_int32(refine_iterations), _p(out["pose"]), _p(out["rms"]), _p(out["n_inliers"]), _p(out["n_hypotheses"]),
        _p(out["status"]), _p(out["assoc"]))
    if st != 0:
        raise ValueError("feo_register_matches: invalid argument")
    return {k: (v[:n] if k == "assoc" else v[:G]) for k, v in out.items()}


def odometry(kp, keypoint_offsets, best, sequence_offsets, window=1, inlier_radius=0.5, min_separation=1.0,
             max_hypotheses=512, min_inliers=16, refine_iterations=4):
    """feo_odometry on the CPU.  kp: (K, 4) float32 keypoints addressed by absolute row; keypoint_offsets (B + 1,);
    best: (ko[B] - ko[1],) int64 (scan s against s - 1); sequence_offsets (S + 1,) in scans.  -> dict of pose, motion
    (B, 4) float64 {c, s, tx, ty}, rms (B,), source, status, n_inliers, n_hypotheses (B,) int32, assoc (ko[B] - ko[0],)
    int64."""
    k = np.ascontiguousarray(kp, np.float32).reshape(-1, 4)
    ko = np.ascontiguousarray(keypoint_offsets, np.int64)
    so = np.ascontiguousarray(sequence_offsets, np.int64)
    B, S = len(ko) - 1, len(so) - 1
    nb = int(ko[-1] - ko[1]) if B >= 2 else 0
    b = np.ascontiguousarray(best, np.int64).reshape(-1)
    assert len(b) == nb, (len(b), nb)
    n = int(ko[-1] - ko[0])
    m = max(B, 1)
    out = {"pose": np.zeros((m, 4)), "motion": np.zeros((m, 4)), "rms": np.zeros(m), "source": np.zeros(m, np.int32),
           "status": np.zeros(m, np.int32), "n_inliers": np.zeros(m, np.int32), "n_hypotheses": np.zeros(m, np.int32),
           "assoc": np.zeros(max(n, 1), np.int64)}
    st = lib().feo_odometry(
        _p(k) if len(k) else None, _p(ko), C.c_int32(B), _p(b) if nb else None, _p(so), C.c_int32(S), C.c_int32(window),
        C.c_double(inlier_radius), C.c_double(min_separation), C.c_int32(max_hypotheses), C.c_int32(min_inliers),
        C.c_int32(refine_iterations), _p(out["pose"]), _p(out["motion"]), _p(out["rms"]), _p(out["source"]),
        _p(out["status"]), _p(out["n_inliers"]), _p(out["n_hypotheses"]), _p(out["assoc"]))
    if st != 0:
        raise ValueError("feo_odometry: invalid argument")
    return {key: (v[:n] if key == "assoc" else v[:B]) for key, v in out.items()}


def loop_closures(kp, descriptors, keypoint_offsets, sequence_offsets, min_gap, candidates, inlier_radius=0.5,
                  min_separation=1.0, max_hypotheses=512, min_inliers=16, refine_iterations=4, n_threads=1):
    """feo_loop_closures on the CPU.  kp: (K, 4) float32 keypoints and descriptors (K, 1980) bins or (K, 1996) records,
    both addressed by absolute row; keypoint_offsets (B + 1,); sequence_offsets (S + 1,) in scans.  -> dict of loop,
    loop_scan (B,) int32, pose (B, 4), rms (B,), n_inliers, n_hypotheses (B,) int32; cand_scan, cand_votes, cand_status,
    cand_inliers, cand_hypotheses (B, candidates) int32, cand_rms (B, candidates), cand_pose (B, candidates, 4); assoc
    (ko[B] - ko[0],) int64."""
    k = np.ascontiguousarray(kp, np.float32).reshape(-1, 4)
    d = np.ascontiguousarray(descriptors, np.float32)
    assert d.ndim == 2 and d.shape[1] in (DESC_LEN, RECORD_FLOATS), d.shape
    first = 5 if d.shape[1] == RECORD_FLOATS else 0
    ko = np.ascontiguousarray(keypoint_offsets, np.int64)
    so = np.ascontiguousarray(sequence_offsets, np.int64)
    B, S = len(ko) - 1, len(so) - 1
    n = int(ko[-1] - ko[0])
    m, K = max(B, 1), max(int(candidates), 1)
    i32 = lambda *sh: np.zeros(sh, np.int32)  # noqa: E731
    out = {"loop": i32(m), "loop_scan": i32(m), "pose": np.zeros((m, 4)), "rms": np.zeros(m), "n_inliers": i32(m),
           "n_hypotheses": i32(m), "cand_scan": i32(m, K), "cand_votes": i32(m, K), "cand_status": i32(m, K),
           "cand_inliers": i32(m, K), "cand_hypotheses": i32(m, K), "cand_rms": np.zeros((m, K)),
           "cand_pose": np.zeros((m, K, 4)), "assoc": np.zeros(max(n, 1), np.int64)}
    st = lib().feo_loop_closures(
        _p(k) if len(k) else None, C.c_void_p(d.ctypes.data + 4 * first if len(d) else None), C.c_int64(d.shape[1]), _p(ko),
        C.c_int32(B), _p(so), C.c_int32(S), C.c_int32(min_gap), C.c_int32(candidates), C.c_double(inlier_radius),
        C.c_double(min_separation), C.c_int32(max_hypotheses), C.c_int32(min_inliers), C.c_int32(refine_iterations),
        C.c_int32(n_threads), *[_p(out[f]) for f in ("loop", "loop_scan", "pose", "rms", "n_inliers", "n_hypotheses",
                                                      "cand_scan", "cand_votes", "cand_status", "cand_inliers",
                                                      "cand_hypotheses", "cand_rms", "cand_pose", "assoc")])
    if st != 0:
        raise ValueError("feo_loop_closures: invalid argument")
    return {key: (v[:n] if key == "assoc" else v[:B]) for key, v in out.items()}
