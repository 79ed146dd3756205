"""fe_register_matches on the B200 against the CPU restatement (match_oracle/fe_register_oracle.cpp), bit for bit: the
pose and rms doubles, the counts, the status and every assoc (include/fe_b200.h, "registration")."""
import ctypes as C
import os

import numpy as np
import pytest

from match_oracle import binding as mo
from register_cases import PARAMS, apply, constructed, oracle_params, relative, sequence
from util import to_fe_params

pytestmark = pytest.mark.gpu

THREADS = len(os.sched_getaffinity(0))


def params(**kw):
    from feature_extraction_b200 import register_params_default
    return register_params_default(**kw)


@pytest.fixture(scope="module")
def node(ob):
    from feature_extraction_b200 import FeatureExtractionNode
    nd = FeatureExtractionNode(to_fe_params(ob.node_default()), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    yield nd
    nd.close()


def assert_same(dev, ora, what=""):
    for k in ("pose", "rms"):
        assert dev[k].shape == ora[k].shape, (what, k)
        assert np.array_equal(dev[k].view(np.uint64), ora[k].view(np.uint64)), (what, k, np.nonzero(dev[k] != ora[k]))
    for k in ("n_inliers", "n_hypotheses", "status", "assoc"):
        assert np.array_equal(dev[k], ora[k]), (what, k, np.nonzero(dev[k] != ora[k])[0][:10])


@pytest.mark.parametrize("kw", [PARAMS, {}, dict(max_hypotheses=7, refine_iterations=0, min_inliers=1)])
def test_constructed_cases_match_the_oracle(node, kw):
    q, r, best, qo, ro, _ = constructed()
    full = dict(inlier_radius=0.5, min_separation=1.0, max_hypotheses=512, min_inliers=16, refine_iterations=4)
    full.update(kw)
    assert_same(node.registerMatches(q, r, best, qo, ro, params(**full)), mo.register_matches(q, r, best, qo, ro, **full))


def _pipeline(ob, synth, cfg, seq):
    from feature_extraction_b200 import FeatureExtractionNode
    pts, offs, rp, poses = sequence(synth, cfg, seq)
    nd = FeatureExtractionNode(to_fe_params(oracle_params(ob, cfg)), max_points=8 << 20, max_scans=64, max_keypoints=1 << 15)
    return nd, pts, offs, rp, poses


@pytest.mark.parametrize("cfg", [1, 2, 4])
def test_real_sequences_scan_to_scan_match_the_oracle(ob, synth, cfg):
    for seq in range(2):
        nd, pts, offs, rp, poses = _pipeline(ob, synth, cfg, seq)
        try:
            ko, kp, d = nd.processBatch(pts, offs, rp)
            qo, ro = ko[1:], ko[:-1]
            for kw in (dict(), dict(min_inliers=3)):
                dev = nd.scan_to_scan(ko, kp, d, params(**kw))
                full = dict(inlier_radius=0.5, min_separation=1.0, max_hypotheses=512, min_inliers=16, refine_iterations=4)
                full.update(kw)
                assert_same(dev, mo.register_matches(kp, kp, dev["best"], qo, ro, **full), (cfg, seq, kw))
        finally:
            nd.close()


def test_scan_against_submap_matches_the_oracle(ob, synth):
    """Groups of one scan against the keypoints of up to 19 previous scans, moved into the scan's frame by the ground
    truth: ~20 queries against ~400 reference rows per group in config 4."""
    nd, pts, offs, rp, poses = _pipeline(ob, synth, 4, 3)
    try:
        ko, kp, d = nd.processBatch(pts, offs, rp)
        world = [np.array([np.cos(p[2]), np.sin(p[2]), p[0], p[1]]) for p in poses]
        Q, R, Dq, Dr, qo, ro = [], [], [], [], [0], [0]
        for s in range(5, len(ko) - 1):
            Q.append(kp[ko[s]:ko[s + 1]])
            Dq.append(d[ko[s]:ko[s + 1]])
            for t in range(max(0, s - 19), s):  # scan t -> scene -> scan s
                rows = kp[ko[t]:ko[t + 1]].copy()
                c, si, x, y = world[s]
                xy = apply(world[t], rows[:, :2]) - [x, y]
                rows[:, 0], rows[:, 1] = c * xy[:, 0] + si * xy[:, 1], -si * xy[:, 0] + c * xy[:, 1]
                R.append(rows)
                Dr.append(d[ko[t]:ko[t + 1]])
            qo.append(qo[-1] + len(Q[-1]))
            ro.append(sum(len(x) for x in R))
        q, r = np.concatenate(Q), np.concatenate(R).astype(np.float32)
        best = nd.matchDescriptors(np.concatenate(Dq), np.concatenate(Dr), qo, ro)[0]
        assert max(np.diff(ro)) >= 300
        for kw in (dict(), dict(min_inliers=3)):
            dev = nd.registerMatches(q, r, best, qo, ro, params(**kw))
            full = dict(inlier_radius=0.5, min_separation=1.0, max_hypotheses=512, min_inliers=16, refine_iterations=4)
            full.update(kw)
            assert_same(dev, mo.register_matches(q, r, best, qo, ro, **full), kw)
        assert (dev["status"] == 2).mean() > 0.5
    finally:
        nd.close()


def test_device_chain_equals_the_host_entry_point(ob, synth):
    """fe_process_batch_device -> fe_match_descriptors_device -> fe_match_device_best -> fe_register_matches_device, with
    no synchronisation in between, gives what the host entry point gives on the downloaded rows."""
    import torch
    nd, pts, offs, rp, poses = _pipeline(ob, synth, 4, 1)
    try:
        dev_pts = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        ko, K, p_kp, p_d = nd.processBatchDevice(dev_pts.data_ptr(), offs, rp)
        best = nd.matchDescriptorsDevice(p_d, 1980, ko[1:], p_d, 1980, ko[:-1])[0]
        p_best = nd.matchDeviceBest()
        dev = nd.registerMatchesDevice(p_kp, p_kp, p_best, ko[1:], ko[:-1], params(min_inliers=3))
        kp = nd.download(p_kp, (K, 4))
        host = nd.registerMatches(kp, kp, best, ko[1:], ko[:-1], params(min_inliers=3))
        assert_same(dev, host)
        assert_same(dev, mo.register_matches(kp, kp, best, ko[1:], ko[:-1], min_inliers=3))
        assert (dev["status"] == 2).mean() > 0.8
        # a register call leaves the match results alone
        assert np.array_equal(nd.download(p_best, (int(ko[-1] - ko[1]),), np.int64), best)
    finally:
        nd.close()


def test_invalid_arguments_leave_the_context_usable(node):
    import torch
    from feature_extraction_b200 import FeatureExtractionError
    from feature_extraction_b200 import _native as N
    q, r, best, qo, ro, _ = constructed()
    good = mo.register_matches(q, r, best, qo, ro, **PARAMS)
    L = N.lib()
    res = N.RegisterResult()

    def call(f, qp, rp, bp, qo_, ro_, G, prm):
        qo_ = np.ascontiguousarray(qo_, np.int64)
        ro_ = np.ascontiguousarray(ro_, np.int64)
        return f(node._ctx, qp, rp, bp, qo_.ctypes.data_as(C.c_void_p), ro_.ctypes.data_as(C.c_void_p), G,
                 C.byref(prm), C.byref(res))
    qp, rp, bp = (q.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p), best.ctypes.data_as(C.c_void_p))
    f = L.fe_register_matches
    P = params(**PARAMS)
    G = len(qo) - 1
    assert call(f, qp, rp, bp, qo, ro, G, P) == N.FE_OK
    assert call(f, qp, rp, bp, qo, ro, -1, P) == N.FE_ERR_INVALID                     # n_groups < 0
    assert call(f, qp, rp, bp, [2, 5, 4], [1, 2, 3], 2, P) == N.FE_ERR_INVALID         # decreasing
    assert call(f, qp, rp, bp, qo, [-1] + list(ro[1:]), G, P) == N.FE_ERR_INVALID      # negative
    assert call(f, None, rp, bp, qo, ro, G, P) == N.FE_ERR_INVALID                     # NULL with rows
    assert call(f, qp, rp, None, qo, ro, G, P) == N.FE_ERR_INVALID
    assert call(f, qp, None, bp, qo, ro, G, P) == N.FE_ERR_INVALID
    for bad in (dict(inlier_radius=0.0), dict(inlier_radius=float("nan")), dict(min_separation=0.0),
                dict(max_hypotheses=0), dict(max_hypotheses=65537), dict(min_inliers=0), dict(refine_iterations=-1)):
        assert call(f, qp, rp, bp, qo, ro, G, params(**bad)) == N.FE_ERR_INVALID, bad
    wrong = best.copy()
    wrong[0] = ro[1]  # a reference row of the next group
    assert call(f, qp, rp, wrong.ctypes.data_as(C.c_void_p), qo, ro, G, P) == N.FE_ERR_INVALID
    with pytest.raises(FeatureExtractionError):
        node.registerMatches(q, r, wrong, qo, ro, P)
    assert_same(node.registerMatches(q, r, best, qo, ro, P), good)
    # the device variant finds a bad `best` on the device
    dq, dr = torch.from_numpy(q).cuda(), torch.from_numpy(r).cuda()
    for b in (wrong, np.where(np.arange(len(best)) == 3, -2, best)):
        db = torch.from_numpy(b).cuda()
        torch.cuda.synchronize()
        st = call(L.fe_register_matches_device, dq.data_ptr(), dr.data_ptr(), db.data_ptr(), qo, ro, G, P)
        assert st == N.FE_ERR_INVALID
    db = torch.from_numpy(best).cuda()
    torch.cuda.synchronize()
    # device keypoints are addressed by absolute row: the arrays hold every row from row 0
    assert_same(node.registerMatchesDevice(dq.data_ptr(), dr.data_ptr(), db.data_ptr(), qo, ro, P), good)
    # empty: n_groups = 0 and a group without rows
    assert node.registerMatches(q, r, best[:0], qo[:1], ro[:1], P)["pose"].shape == (0, 4)
