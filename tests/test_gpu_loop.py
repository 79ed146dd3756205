"""fe_loop_closures on the B200 against the CPU restatement (match_oracle/fe_loop_oracle.cpp), bit for bit: every pose
and rms double, the votes, counts, status and every assoc (include/fe_b200.h, "loop closures")."""
import ctypes as C
import os

import numpy as np
import pytest

from loop_cases import constructed, loop_sequence, oracle_chain
from match_oracle import binding as mo
from register_cases import kp as make_kp, oracle_params
from util import to_fe_params

pytestmark = pytest.mark.gpu

THREADS = len(os.sched_getaffinity(0))
FLOATS = ("pose", "rms", "cand_rms", "cand_pose")
INTS = ("loop", "loop_scan", "n_inliers", "n_hypotheses", "cand_scan", "cand_votes", "cand_status", "cand_inliers",
        "cand_hypotheses", "assoc")


def lp(min_gap, candidates):
    from feature_extraction_b200 import loop_params_default
    return loop_params_default(min_gap=min_gap, candidates=candidates)


def rp(**kw):
    from feature_extraction_b200 import register_params_default
    return register_params_default(**kw)


@pytest.fixture(scope="module")
def node(ob):
    from feature_extraction_b200 import FeatureExtractionNode
    nd = FeatureExtractionNode(to_fe_params(ob.node_default()), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    yield nd
    nd.close()


def assert_same(dev, ora, what=""):
    for k in FLOATS:
        assert dev[k].shape == ora[k].shape, (what, k)
        assert np.array_equal(dev[k].view(np.uint64), ora[k].view(np.uint64)), (what, k, np.nonzero(dev[k] != ora[k]))
    for k in INTS:
        assert dev[k].shape == ora[k].shape, (what, k)
        assert np.array_equal(dev[k], ora[k]), (what, k, np.argwhere(dev[k] != ora[k])[:10])


def test_constructed_sequences_match_the_oracle(node):
    kp, d, ko, so, cases, _ = constructed()
    for c in cases:
        for K in sorted({c["candidates"], 1, 16}):
            for kw in ({}, dict(min_inliers=3, max_hypotheses=7, refine_iterations=0)):
                dev = node.loopClosures(kp, d, ko, so, lp(c["min_gap"], K), rp(**kw))
                assert_same(dev, mo.loop_closures(kp, d, ko, so, c["min_gap"], K, **kw), (c["scans"], K, kw))
                assert node.last_launches <= 9


def _batch(chains, lengths):
    """Oracle chains cut to the given lengths, concatenated into one batch -> kp, descriptors, ko, so."""
    K, D, KO, SO = [], [], [0], [0]
    for (cfg, kind, seq), n in zip(chains, lengths):
        ko, kp, d, _ = oracle_chain(cfg, kind, seq)
        ko = ko[:n + 1]
        K.append(kp[ko[0]:ko[-1]])
        D.append(d[ko[0]:ko[-1]])
        KO.extend((ko[1:] - ko[0] + KO[-1]).tolist())
        SO.append(len(KO) - 1)
    return np.concatenate(K), np.concatenate(D), np.array(KO, np.int64), np.array(SO, np.int64)


@pytest.mark.parametrize("cfg", [2, 4])
def test_loop_sequences_match_the_oracle(node, cfg):
    kp, d, ko, so = _batch([(cfg, "loop", 0), (cfg, "loop", 1), (cfg, "forward", 0)], [30, 30, 20])
    found = 0
    for gap, K, kw in ((3, 1, {}), (3, 4, {}), (10, 1, {}), (10, 4, {}), (3, 4, dict(min_inliers=3))):
        dev = node.loopClosures(kp, d, ko, so, lp(gap, K), rp(**kw))
        assert_same(dev, mo.loop_closures(kp, d, ko, so, gap, K, n_threads=THREADS, **kw), (gap, K, kw))
        found += int((dev["loop"] >= 0).sum())
    assert found > 0


def test_sequences_of_unequal_length_in_one_batch(node):
    kp, d, ko, so = _batch([(4, "loop", 2), (4, "loop", 3), (2, "loop", 4), (4, "forward", 1), (4, "loop", 5)],
                           [30, 7, 12, 0, 1])
    assert list(np.diff(so)) == [30, 7, 12, 0, 1]
    for gap, K in ((1, 2), (5, 3), (40, 1)):
        assert_same(node.loopClosures(kp, d, ko, so, lp(gap, K)), mo.loop_closures(kp, d, ko, so, gap, K, n_threads=THREADS),
                    (gap, K))


def test_a_database_longer_than_one_segment(node):
    """Scan 0 holds 1,100 rows, so the retrieval of scans 1 and 2 (min_gap 1) and every verification against scan 0 run
    in two segments each, with k_match_merge; scan 2 repeats 60 of scan 0's rows and registers against it."""
    rng = np.random.default_rng(11)
    n0 = 1100
    xy0 = rng.uniform(-60.0, 60.0, (n0, 2)).round(1)
    d0 = rng.random((n0, 1980), dtype=np.float32)
    pick = rng.choice(n0, 60, replace=False)
    kp = np.concatenate([make_kp(xy0), make_kp(rng.uniform(-60.0, 60.0, (50, 2))), make_kp(xy0[pick])])
    d = np.concatenate([d0, rng.random((50, 1980), dtype=np.float32), d0[pick]])
    ko = np.array([0, n0, n0 + 50, n0 + 110], np.int64)
    so = np.array([0, 3], np.int64)
    for K in (1, 3):
        dev = node.loopClosures(kp, d, ko, so, lp(1, K))
        assert_same(dev, mo.loop_closures(kp, d, ko, so, 1, K, n_threads=THREADS), K)
        assert dev["loop_scan"][2] == 0 and dev["n_inliers"][2] == 60
        assert node.last_launches == 9


def test_device_chain_equals_the_host_entry_point(ob, synth):
    """fe_process_batch_device -> fe_loop_closures_device, with no synchronisation in between, gives what the host
    entry point gives on the downloaded rows."""
    import torch
    from feature_extraction_b200 import FeatureExtractionNode
    pts, offs, rp_, _ = loop_sequence(synth, 4, 6)
    nd = FeatureExtractionNode(to_fe_params(oracle_params(ob, 4)), max_points=8 << 20, max_scans=64, max_keypoints=1 << 15)
    try:
        dev_pts = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        ko, K, p_kp, p_d = nd.processBatchDevice(dev_pts.data_ptr(), offs, rp_)
        so = [0, 22, len(ko) - 1]
        dev = nd.loopClosuresDevice(p_kp, p_d, 1980, ko, so)
        kp = nd.download(p_kp, (K, 4))
        d = nd.download(p_d, (K, 1980))
        assert_same(dev, nd.sequence_loop_closures(ko, kp, d, so))
        from feature_extraction_b200 import loop_params_default
        p = loop_params_default()
        assert_same(dev, mo.loop_closures(kp, d, ko, so, p.min_gap, p.candidates, n_threads=THREADS))
        assert (dev["loop"] >= 0).sum() >= 1
    finally:
        nd.close()


def test_loop_results_and_the_other_calls_leave_each_other_alone(node):
    """The host results of a loop-closure call survive match, register and odometry calls, and theirs survive it."""
    from feature_extraction_b200 import _native as N
    from feature_extraction_b200.node import _unpack_loop, _unpack_match, _unpack_odometry, _unpack_register
    from match_cases import random_rows
    from odometry_cases import constructed as odo_case, scan_pairs_best
    rng = np.random.default_rng(3)
    kp, d, ko, so, cases, _ = constructed()
    loop_res = N.LoopResult()
    lp_, rp_ = lp(2, 4), rp()
    k_ = np.ascontiguousarray(kp)
    d_ = np.ascontiguousarray(d)
    assert N.lib().fe_loop_closures(node._ctx, k_.ctypes.data_as(C.c_void_p), d_.ctypes.data_as(C.c_void_p), 1980,
                                    ko.ctypes.data_as(C.c_void_p), len(ko) - 1, so.ctypes.data_as(C.c_void_p), len(so) - 1,
                                    C.byref(lp_), C.byref(rp_), C.byref(loop_res)) == N.FE_OK
    loop_before = _unpack_loop(loop_res)
    okp, oko, obest, oso, _, _ = odo_case()
    q, r = random_rows(rng, 40), random_rows(rng, 300)
    m_res = N.MatchResult()
    qo, ro = np.array([0, 40], np.int64), np.array([0, 300], np.int64)
    assert N.lib().fe_match_descriptors(node._ctx, q.ctypes.data_as(C.c_void_p), 1980, qo.ctypes.data_as(C.c_void_p),
                                        r.ctypes.data_as(C.c_void_p), 1980, ro.ctypes.data_as(C.c_void_p), 1,
                                        C.byref(m_res)) == N.FE_OK
    match_before = _unpack_match(m_res)
    reg_res = N.RegisterResult()
    b = scan_pairs_best(oko, obest, oso)
    rqo, rro = oko[1:].copy(), oko[:-1].copy()
    assert N.lib().fe_register_matches(node._ctx, okp.ctypes.data_as(C.c_void_p), okp.ctypes.data_as(C.c_void_p),
                                       b.ctypes.data_as(C.c_void_p), rqo.ctypes.data_as(C.c_void_p),
                                       rro.ctypes.data_as(C.c_void_p), len(rqo) - 1, C.byref(rp_), C.byref(reg_res)) == N.FE_OK
    reg_before = _unpack_register(reg_res)
    odo_res = N.OdometryResult()
    assert N.lib().fe_odometry(node._ctx, okp.ctypes.data_as(C.c_void_p), oko.ctypes.data_as(C.c_void_p), len(oko) - 1,
                               obest.ctypes.data_as(C.c_void_p), oso.ctypes.data_as(C.c_void_p), len(oso) - 1, 2,
                               C.byref(rp_), C.byref(odo_res)) == N.FE_OK
    odo_before = _unpack_odometry(odo_res)
    assert_same(_unpack_loop(loop_res), loop_before)  # the loop results survive match, register and odometry calls
    # a larger loop-closure call, which grows the loop buffers: the other results survive it
    kp4, d4, ko4, so4 = _batch([(4, "loop", 0)], [30])
    node.loopClosures(kp4, d4, ko4, so4, lp(3, 8))
    assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(_unpack_match(m_res), match_before))
    for now, before in ((_unpack_register(reg_res), reg_before), (_unpack_odometry(odo_res), odo_before)):
        assert all(np.array_equal(now[k].view(np.uint8), before[k].view(np.uint8)) for k in before)
    assert_same(loop_before, mo.loop_closures(kp, d, ko, so, 2, 4))


def test_invalid_arguments_leave_the_context_usable(node):
    import torch
    from feature_extraction_b200 import FeatureExtractionError
    from feature_extraction_b200 import _native as N
    kp, d, ko, so, _, _ = constructed()
    good = mo.loop_closures(kp, d, ko, so, 2, 3)
    L = N.lib()
    res = N.LoopResult()

    def call(f, kpp, dp, stride, ko_, B, so_, S, lpar, prm):
        ko_ = np.ascontiguousarray(ko_, np.int64)
        so_ = np.ascontiguousarray(so_, np.int64)
        return f(node._ctx, kpp, dp, stride, ko_.ctypes.data_as(C.c_void_p), B, so_.ctypes.data_as(C.c_void_p), S,
                 lpar, prm, C.byref(res))
    kpp, dp = kp.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p)
    f = L.fe_loop_closures
    B, S = len(ko) - 1, len(so) - 1
    P, Q = C.byref(lp(2, 3)), C.byref(rp())
    assert call(f, kpp, dp, 1980, ko, B, so, S, P, Q) == N.FE_OK
    assert call(f, kpp, dp, 1980, ko, -1, so, S, P, Q) == N.FE_ERR_INVALID                        # n_scans < 0
    assert call(f, kpp, dp, 1980, ko, B, so, -1, P, Q) == N.FE_ERR_INVALID                        # n_sequences < 0
    assert call(f, kpp, dp, 1979, ko, B, so, S, P, Q) == N.FE_ERR_INVALID                         # stride
    for gap, K in ((0, 3), (-1, 3), (2, 0), (2, 17)):
        assert call(f, kpp, dp, 1980, ko, B, so, S, C.byref(lp(gap, K)), Q) == N.FE_ERR_INVALID, (gap, K)
    bad_ko = ko.copy()
    bad_ko[3] = bad_ko[2] - 1
    assert call(f, kpp, dp, 1980, bad_ko, B, so, S, P, Q) == N.FE_ERR_INVALID                    # decreasing
    assert call(f, kpp, dp, 1980, [-1] + list(ko[1:]), B, so, S, P, Q) == N.FE_ERR_INVALID        # negative
    assert call(f, kpp, dp, 1980, ko, B, [1] + list(so[1:]), S, P, Q) == N.FE_ERR_INVALID         # does not start at 0
    assert call(f, kpp, dp, 1980, ko, B, list(so[:-1]) + [B - 1], S, P, Q) == N.FE_ERR_INVALID    # does not end at B
    assert call(f, kpp, dp, 1980, ko, B, [0, 5, 3, B], 3, P, Q) == N.FE_ERR_INVALID               # decreasing
    big = np.array([0, 1 << 24], np.int64)
    assert call(f, kpp, dp, 1980, big, 1, [0, 1], 1, P, Q) == N.FE_ERR_INVALID                    # 2^24 rows in a scan
    assert call(f, None, dp, 1980, ko, B, so, S, P, Q) == N.FE_ERR_INVALID                        # NULL with rows
    assert call(f, kpp, None, 1980, ko, B, so, S, P, Q) == N.FE_ERR_INVALID
    assert f(node._ctx, kpp, dp, 1980, None, B, so.ctypes.data_as(C.c_void_p), S, P, Q, C.byref(res)) == N.FE_ERR_INVALID
    assert call(f, kpp, dp, 1980, ko, B, so, S, None, Q) == N.FE_ERR_INVALID                      # loop_params NULL
    assert call(f, kpp, dp, 1980, ko, B, so, S, P, None) == N.FE_ERR_INVALID                      # params NULL
    for bad in (dict(inlier_radius=0.0), dict(inlier_radius=float("nan")), dict(min_separation=0.0),
                dict(max_hypotheses=0), dict(max_hypotheses=65537), dict(min_inliers=0), dict(refine_iterations=-1),
                dict(refine_iterations=1001)):
        assert call(f, kpp, dp, 1980, ko, B, so, S, P, C.byref(rp(**bad))) == N.FE_ERR_INVALID, bad
    with pytest.raises(FeatureExtractionError):
        node.loopClosures(kp, d, ko, so, lp(0, 3))
    with pytest.raises(ValueError):
        node.loopClosures(kp, d, ko, so[:-1], lp(2, 3))
    assert_same(node.loopClosures(kp, d, ko, so, lp(2, 3)), good)
    dk, dd = torch.from_numpy(kp).cuda(), torch.from_numpy(d).cuda()
    torch.cuda.synchronize()
    assert call(L.fe_loop_closures_device, dk.data_ptr(), None, 1980, ko, B, so, S, P, Q) == N.FE_ERR_INVALID
    assert_same(node.loopClosuresDevice(dk.data_ptr(), dd.data_ptr(), 1980, ko, so, lp(2, 3)), good)
    # empty: no scans, and no eligible scans
    e = node.loopClosures(kp[:0], d[:0], [0], [0])
    assert e["pose"].shape == (0, 4) and node.last_launches == 0
    one = node.loopClosures(kp[:0], d[:0], [0, 0], [0, 0, 1, 1], lp(1, 2))
    assert list(one["loop"]) == [-1] and one["cand_scan"].tolist() == [[-1, -1]] and node.last_launches == 1
