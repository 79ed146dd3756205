"""fe_odometry on the B200 against the CPU restatement (match_oracle/fe_odometry_oracle.cpp), bit for bit: the pose,
motion and rms doubles, the counts, source, status and every assoc (include/fe_b200.h, "odometry")."""
import ctypes as C
import os

import numpy as np
import pytest

from match_oracle import binding as mo
from odometry_cases import constructed, oracle_chain, scan_pairs_best
from register_cases import oracle_params, sequence
from util import bits_equal, to_fe_params

pytestmark = pytest.mark.gpu

THREADS = len(os.sched_getaffinity(0))
FIELDS = ("pose", "motion", "rms", "n_inliers", "n_hypotheses", "source", "status", "assoc")


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
    for k in ("pose", "motion", "rms"):
        assert dev[k].shape == ora[k].shape, (what, k)
        assert np.array_equal(dev[k].view(np.uint64), ora[k].view(np.uint64)), (what, k, np.nonzero(dev[k] != ora[k]))
    for k in ("n_inliers", "n_hypotheses", "source", "status", "assoc"):
        assert np.array_equal(dev[k], ora[k]), (what, k, np.nonzero(dev[k] != ora[k])[0][:10])


@pytest.mark.parametrize("W", [1, 2, 4, 64])
def test_constructed_sequences_match_the_oracle(node, W):
    kp, ko, best, so, _, _ = constructed()
    for kw in ({}, dict(min_inliers=3, max_hypotheses=7, refine_iterations=0)):
        dev = node.odometry(kp, ko, best, so, W, params(**kw))
        assert_same(dev, mo.odometry(kp, ko, best, so, W, **kw), (W, kw))


def _batch(cfgs_seqs, n_scans):
    """Oracle chains of several sequences, each cut to its own length, concatenated into one batch -> kp, ko, best, so.
    `best` of a first scan keeps what a matcher of scan s against s - 1 would give it: rows of the previous sequence."""
    K, KO, B, SO = [], [0], [], [0]
    for (cfg, seq), n in zip(cfgs_seqs, n_scans):
        ko, kp, best, _ = oracle_chain(cfg, seq)
        ko = ko[:n + 1]
        shift = KO[-1] - ko[0]
        first = np.full(ko[1] - ko[0], -1 if KO[-1] == 0 else KO[-1] - 1, np.int64)
        if len(KO) > 1:
            B.append(first)
        B.append(np.where(best[:ko[-1] - ko[1]] < 0, -1, best[:ko[-1] - ko[1]] + shift))
        K.append(kp[ko[0]:ko[-1]])
        KO.extend((ko[1:] + shift).tolist())
        SO.append(len(KO) - 1)
    return np.concatenate(K), np.array(KO, np.int64), np.concatenate(B), np.array(SO, np.int64)


@pytest.mark.parametrize("cfg", [2, 4])
def test_real_sequences_match_the_oracle(node, cfg):
    from feature_extraction_b200 import ODOMETRY_WINDOW
    kp, ko, best, so = _batch([(cfg, i) for i in range(4)], [20] * 4)
    for W in sorted({1, 2, ODOMETRY_WINDOW, 8}):
        for kw in ({}, dict(min_inliers=3)):
            assert_same(node.odometry(kp, ko, best, so, W, params(**kw)), mo.odometry(kp, ko, best, so, W, **kw), (W, kw))


def test_sequences_of_unequal_length_in_one_batch(node):
    kp, ko, best, so = _batch([(4, 5), (4, 6), (2, 7), (4, 8)], [20, 3, 11, 1])
    assert list(np.diff(so)) == [20, 3, 11, 1]
    for W in (1, 3, 8):
        dev = node.odometry(kp, ko, best, so, W, params(min_inliers=3))
        assert_same(dev, mo.odometry(kp, ko, best, so, W, min_inliers=3), W)
        assert node.last_launches == 1 + 3 * 19


def test_window_one_equals_scan_to_scan(ob, synth):
    from feature_extraction_b200 import FeatureExtractionNode
    pts, offs, rp, _ = sequence(synth, 4, 2)
    nd = FeatureExtractionNode(to_fe_params(oracle_params(ob, 4)), max_points=8 << 20, max_scans=64, max_keypoints=1 << 15)
    try:
        ko, kp, d = nd.processBatch(pts, offs, rp)
        so = [0, 7, 7, len(ko) - 1]  # two sequences and an empty one
        for kw in ({}, dict(min_inliers=3)):
            s2s = nd.scan_to_scan(ko, kp, d, params(**kw))
            odo = nd.sequence_odometry(ko, kp, d, so, 1, params(**kw))
            assert np.array_equal(odo["best"], s2s["best"])
            for s in range(1, len(ko) - 1):
                if s == 7:
                    continue
                g = s - 1
                for k in ("status", "n_inliers", "n_hypotheses"):
                    assert odo[k][s] == s2s[k][g], (s, k)
                assert odo["rms"][s].view(np.uint64) == s2s["rms"][g].view(np.uint64)
                if s2s["status"][g] == 2:
                    assert np.array_equal(odo["motion"][s].view(np.uint64), s2s["pose"][g].view(np.uint64))
                assert np.array_equal(odo["assoc"][ko[s]:ko[s + 1]], s2s["assoc"][ko[s] - ko[1]:ko[s + 1] - ko[1]])
            assert_same(odo, mo.odometry(kp, ko, odo["best"], so, 1, **{"min_inliers": 16, **kw}))
    finally:
        nd.close()


def test_device_chain_equals_the_host_entry_point(ob, synth):
    """fe_process_batch_device -> fe_match_descriptors_device -> fe_match_device_best -> fe_odometry_device, with no
    synchronisation in between, gives what the host entry point gives on the downloaded rows."""
    import torch
    from feature_extraction_b200 import FeatureExtractionNode, ODOMETRY_WINDOW
    pts, offs, rp, _ = sequence(synth, 4, 1)
    nd = FeatureExtractionNode(to_fe_params(oracle_params(ob, 4)), max_points=8 << 20, max_scans=64, max_keypoints=1 << 15)
    try:
        dev_pts = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        ko, K, p_kp, p_d = nd.processBatchDevice(dev_pts.data_ptr(), offs, rp)
        best = nd.matchDescriptorsDevice(p_d, 1980, ko[1:], p_d, 1980, ko[:-1])[0]
        p_best = nd.matchDeviceBest()
        so = [0, 12, len(ko) - 1]
        dev = nd.odometryDevice(p_kp, ko, p_best, so, ODOMETRY_WINDOW)
        kp = nd.download(p_kp, (K, 4))
        assert_same(dev, nd.odometry(kp, ko, best, so, ODOMETRY_WINDOW))
        assert_same(dev, mo.odometry(kp, ko, best, so, ODOMETRY_WINDOW))
        assert (dev["source"] == 1).sum() >= 10
        # an odometry call leaves the match results alone
        assert np.array_equal(nd.download(p_best, (int(ko[-1] - ko[1]),), np.int64), best)
    finally:
        nd.close()


def test_register_and_odometry_results_leave_each_other_alone(node):
    """The host results of a match, a register and an odometry call each survive the other two kinds of call."""
    from feature_extraction_b200 import _native as N
    from match_cases import constructed as match_case, random_rows
    rng = np.random.default_rng(25)
    mq, mr, mqo, mro = match_case(rng)
    m_res = N.MatchResult()
    assert N.lib().fe_match_descriptors(node._ctx, mq.ctypes.data_as(C.c_void_p), mq.shape[1], mqo.ctypes.data_as(C.c_void_p),
                                        mr.ctypes.data_as(C.c_void_p), mr.shape[1], mro.ctypes.data_as(C.c_void_p),
                                        len(mqo) - 1, C.byref(m_res)) == N.FE_OK
    from feature_extraction_b200.node import _unpack_match, _unpack_odometry, _unpack_register
    match_before = _unpack_match(m_res)
    same_match = lambda a, b_: all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b_))  # noqa: E731
    kp, ko, best, so, _, _ = constructed()
    b = scan_pairs_best(ko, best, so)
    res = N.RegisterResult()
    prm = params()
    qo, ro = ko[1:].copy(), ko[:-1].copy()
    assert N.lib().fe_register_matches(node._ctx, kp.ctypes.data_as(C.c_void_p), kp.ctypes.data_as(C.c_void_p),
                                       b.ctypes.data_as(C.c_void_p), qo.ctypes.data_as(C.c_void_p),
                                       ro.ctypes.data_as(C.c_void_p), len(qo) - 1, C.byref(prm), C.byref(res)) == N.FE_OK
    reg_before = _unpack_register(res)
    assert same_match(_unpack_match(m_res), match_before)  # the match results survive a register call
    odo_res = N.OdometryResult()
    so_ = so.copy()
    assert N.lib().fe_odometry(node._ctx, kp.ctypes.data_as(C.c_void_p), ko.ctypes.data_as(C.c_void_p), len(ko) - 1,
                               best.ctypes.data_as(C.c_void_p), so_.ctypes.data_as(C.c_void_p), len(so_) - 1, 2,
                               C.byref(prm), C.byref(odo_res)) == N.FE_OK
    odo_before = _unpack_odometry(odo_res)
    assert_reg = lambda a, b_: all(np.array_equal(a[k], b_[k]) for k in a)  # noqa: E731
    assert assert_reg(_unpack_register(res), reg_before)  # the register results survive an odometry call
    assert same_match(_unpack_match(m_res), match_before)  # and so do the match results
    node.registerMatches(kp, kp, b, qo, ro)
    assert_same(_unpack_odometry(odo_res), odo_before)  # and the odometry results a register call
    # a larger match call, which grows the match buffers: the register and odometry results survive it
    node.matchDescriptors(random_rows(rng, 300), random_rows(rng, 2000))
    assert assert_reg(_unpack_register(res), reg_before)
    assert_same(_unpack_odometry(odo_res), odo_before)
    assert_same(odo_before, mo.odometry(kp, ko, best, so, 2))
    assert assert_reg(reg_before, mo.register_matches(kp, kp, b, qo, ro))
    m_ora = mo.match_descriptors(mq, mr, mqo, mro)
    assert all(np.array_equal(x, y) for x, y in zip(match_before[:2], m_ora[:2]))
    assert all(bits_equal(x, y) for x, y in zip(match_before[2:], m_ora[2:]))


def test_invalid_arguments_leave_the_context_usable(node):
    import torch
    from feature_extraction_b200 import FeatureExtractionError
    from feature_extraction_b200 import _native as N
    kp, ko, best, so, _, _ = constructed()
    good = mo.odometry(kp, ko, best, so, 2)
    L = N.lib()
    res = N.OdometryResult()

    def call(f, kpp, ko_, B, bp, so_, S, W, prm):
        ko_ = np.ascontiguousarray(ko_, np.int64)
        so_ = np.ascontiguousarray(so_, np.int64)
        return f(node._ctx, kpp, ko_.ctypes.data_as(C.c_void_p), B, bp, so_.ctypes.data_as(C.c_void_p), S, W,
                 C.byref(prm), C.byref(res))
    kpp, bp = kp.ctypes.data_as(C.c_void_p), best.ctypes.data_as(C.c_void_p)
    f = L.fe_odometry
    P = params()
    B, S = len(ko) - 1, len(so) - 1
    assert call(f, kpp, ko, B, bp, so, S, 2, P) == N.FE_OK
    assert call(f, kpp, ko, -1, bp, so, S, 2, P) == N.FE_ERR_INVALID                        # n_scans < 0
    assert call(f, kpp, ko, B, bp, so, -1, 2, P) == N.FE_ERR_INVALID                        # n_sequences < 0
    for W in (0, 65):
        assert call(f, kpp, ko, B, bp, so, S, W, P) == N.FE_ERR_INVALID                     # window
    bad_ko = ko.copy()
    bad_ko[3] = bad_ko[2] - 1
    assert call(f, kpp, bad_ko, B, bp, so, S, 2, P) == N.FE_ERR_INVALID                    # decreasing
    assert call(f, kpp, [-1] + list(ko[1:]), B, bp, so, S, 2, P) == N.FE_ERR_INVALID        # negative
    assert call(f, kpp, ko, B, bp, [1] + list(so[1:]), S, 2, P) == N.FE_ERR_INVALID         # does not start at 0
    assert call(f, kpp, ko, B, bp, list(so[:-1]) + [B - 1], S, 2, P) == N.FE_ERR_INVALID    # does not end at B
    assert call(f, kpp, ko, B, bp, [0, 5, 3, B], 3, 2, P) == N.FE_ERR_INVALID               # decreasing
    assert call(f, None, ko, B, bp, so, S, 2, P) == N.FE_ERR_INVALID                        # NULL with rows
    assert call(f, kpp, ko, B, None, so, S, 2, P) == N.FE_ERR_INVALID
    assert f(node._ctx, kpp, None, B, bp, so.ctypes.data_as(C.c_void_p), S, 2, C.byref(P), C.byref(res)) == N.FE_ERR_INVALID
    assert f(node._ctx, kpp, ko.ctypes.data_as(C.c_void_p), B, bp, so.ctypes.data_as(C.c_void_p), S, 2, None,
             C.byref(res)) == N.FE_ERR_INVALID                                             # params NULL
    for bad in (dict(inlier_radius=0.0), dict(inlier_radius=float("nan")), dict(min_separation=0.0),
                dict(max_hypotheses=0), dict(max_hypotheses=65537), dict(min_inliers=0), dict(refine_iterations=-1),
                dict(refine_iterations=1001)):
        assert call(f, kpp, ko, B, bp, so, S, 2, params(**bad)) == N.FE_ERR_INVALID, bad
    wrong = best.copy()
    wrong[ko[2] - ko[1]] = ko[0]  # scan 2's row into scan 0: not the previous scan
    assert call(f, kpp, ko, B, wrong.ctypes.data_as(C.c_void_p), so, S, 2, P) == N.FE_ERR_INVALID
    with pytest.raises(FeatureExtractionError):
        node.odometry(kp, ko, wrong, so, 2)
    with pytest.raises(ValueError):
        node.odometry(kp, ko, best[:-1], so, 2)
    with pytest.raises(ValueError):
        node.odometry(kp, ko, best, so[:-1], 2)
    assert_same(node.odometry(kp, ko, best, so, 2), good)
    # the device variant finds a bad `best` on the device
    dk = torch.from_numpy(kp).cuda()
    for b in (wrong, np.where(np.arange(len(best)) == ko[4] - ko[1], -2, best)):
        db = torch.from_numpy(b).cuda()
        torch.cuda.synchronize()
        assert call(L.fe_odometry_device, dk.data_ptr(), ko, B, db.data_ptr(), so, S, 2, P) == N.FE_ERR_INVALID
    db = torch.from_numpy(best).cuda()
    torch.cuda.synchronize()
    assert_same(node.odometryDevice(dk.data_ptr(), ko, db.data_ptr(), so, 2), good)
    # empty: no scans, and scans without sequences of two
    e = node.odometry(kp[:0], [0], np.zeros(0, np.int64), [0], 2)
    assert e["pose"].shape == (0, 4) and node.last_launches == 0
    one = node.odometry(kp[:0], [0, 0], np.zeros(0, np.int64), [0, 0, 1, 1], 2)
    assert list(one["source"]) == [0] and list(one["status"]) == [-1]
