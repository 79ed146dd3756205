"""fe_match_descriptors on the B200 against the CPU oracle (match_oracle/fe_match_oracle.cpp), element for element:
best, shift and the bits of dist2 / second_dist2 (include/fe_b200.h, "descriptor matching")."""
import ctypes as C
import os

import numpy as np
import pytest

from match_oracle import binding as mo
from match_cases import constructed, random_rows, rolled, to_records
from util import bits_equal, to_fe_params

pytestmark = pytest.mark.gpu

THREADS = len(os.sched_getaffinity(0))


def _params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


@pytest.fixture(scope="module")
def node(ob):
    from feature_extraction_b200 import FeatureExtractionNode
    nd = FeatureExtractionNode(to_fe_params(ob.node_default()), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    yield nd
    nd.close()


def assert_same(dev, ora, what=""):
    best, shift, d, sd = dev
    ob_, os_, od, osd = ora
    assert len(best) == len(ob_), what
    assert np.array_equal(best, ob_), (what, np.nonzero(best != ob_)[0][:10])
    assert np.array_equal(shift, os_), (what, np.nonzero(shift != os_)[0][:10])
    assert bits_equal(d, od), (what, np.nonzero(d.view(np.uint32) != od.view(np.uint32))[0][:10])
    assert bits_equal(sd, osd), (what, np.nonzero(sd.view(np.uint32) != osd.view(np.uint32))[0][:10])


@pytest.mark.parametrize("cfg", [1, 2, 3, 4])
def test_real_descriptors_match_the_oracle(ob, synth, cfg):
    from feature_extraction_b200 import FeatureExtractionNode
    nd = FeatureExtractionNode(to_fe_params(_params(ob, cfg)), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    try:
        pts, offs, rp = synth.generate(cfg, 12, scan_index_base=40)
        ko, kp, d = nd.processBatch(pts, offs, rp)
        assert len(d) > 0
        # scan s against scan s - 1
        qo, ro = ko[1:], ko[:-1]
        assert_same(nd.matchDescriptors(d, d, qo, ro), mo.match_descriptors(d, d, qo, ro, n_threads=THREADS), "s vs s-1")
        # everything against everything, one group (at most 600 rows)
        n = min(len(d), 600)
        dev = nd.matchDescriptors(d[:n], d[:n])
        assert_same(dev, mo.match_descriptors(d[:n], d[:n], n_threads=THREADS), "all vs all")
        fin = np.isfinite(d[:n]).all(axis=1)
        assert (dev[0][fin] <= np.arange(n)[fin]).all() and (dev[2][fin] == 0).all()
    finally:
        nd.close()


def test_constructed_cases_match_the_oracle(ob, node):
    rng = np.random.default_rng(21)
    q, r, qo, ro = constructed(rng)
    dev = node.matchDescriptors(q, r, qo, ro)
    assert_same(dev, mo.match_descriptors(q, r, qo, ro))
    best, shift, d, sd = dev
    assert best[1] == 3 and shift[1] == 5 and d[1] == 0.0
    assert best[2] == 6 and sd[2] == 0.0 and best[7] == 12 and best[10] == 17 and sd[10] == d[10]
    assert (best[3:6] == -1).all() and np.isposinf(d[3:6]).all() and np.isposinf(sd[3:6]).all()
    # G = 0, and a group with queries only
    assert all(len(a) == 0 for a in node.matchDescriptors(q, r, [2], [4]))
    b2 = node.matchDescriptors(q, r, [0, 3], [5, 5])
    assert (b2[0] == -1).all() and (b2[1] == -1).all() and np.isposinf(b2[2]).all() and np.isposinf(b2[3]).all()


def test_tile_edges_of_both_sides(ob, node):
    """Groups of 1, 31, 32, 33 and 257 rows on either side, every combination, with planted rolled copies."""
    rng = np.random.default_rng(22)
    sizes = [1, 31, 32, 33, 257]
    qo, ro = [0], [0]
    for a in sizes:
        for b in sizes:
            qo.append(qo[-1] + a)
            ro.append(ro[-1] + b)
    q = random_rows(rng, qo[-1])
    r = random_rows(rng, ro[-1])
    for g in range(len(sizes) ** 2):  # the last query of a group rolled into the last reference row of the group
        r[ro[g + 1] - 1] = rolled(q[qo[g + 1] - 1], g % 12)
    dev = node.matchDescriptors(q, r, qo, ro)
    assert_same(dev, mo.match_descriptors(q, r, qo, ro, n_threads=THREADS))
    last = np.array(qo[1:]) - 1
    assert np.array_equal(dev[0][last], np.array(ro[1:]) - 1) and (dev[2][last] == 0).all()


def test_one_large_group_crosses_every_segment_merge(ob, node):
    """About 2,000 x 20,000 rows in one group: the reference side is cut into segments and merged; the oracle checks a
    sample of queries against all 20,000 reference rows (a query's result depends only on its group)."""
    rng = np.random.default_rng(23)
    nq, nr = 2003, 20011
    q = random_rows(rng, nq)
    r = random_rows(rng, nr)
    q[700] = np.nan
    # ties across the segment boundary at 1024 and far apart: the lower row wins, second == best
    for k in (1023, 1024, 15000):
        r[k] = rolled(q[5], 4)
    r[19999] = rolled(q[1999], 9)
    r[3] = rolled(q[2002], 0)
    dev = node.matchDescriptors(q, r)
    best, shift, d, sd = dev
    assert best[5] == 1023 and shift[5] == 4 and d[5] == 0.0 and sd[5] == 0.0
    assert best[1999] == 19999 and shift[1999] == 9 and best[2002] == 3 and best[700] == -1
    sample = np.array([0, 1, 2, 3, 4, 5, 6, 7, 700, 1022, 1023, 1024, 1025, 1999, 2000, 2002])
    ora = mo.match_descriptors(q[sample], r, n_threads=THREADS)
    assert_same(tuple(a[sample] for a in dev), ora)


def test_record_output_equals_plain_bins(ob, synth):
    from feature_extraction_b200 import FeatureExtractionNode
    nd = FeatureExtractionNode(to_fe_params(ob.node_default()), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    try:
        pts, offs, rp = synth.generate(2, 20, scan_index_base=90)
        ko, kp, d = nd.processBatch(pts, offs, rp)
        nd.enableRecordOutput(True)
        ko2, kp2, rec = nd.processBatch(pts, offs, rp)
        assert rec.shape == (len(d), 1996) and bits_equal(rec[:, 5:1985], d)
        a = nd.matchDescriptors(d, d, ko[1:], ko[:-1])
        b = nd.matchDescriptors(rec, rec, ko[1:], ko[:-1])
        c = nd.matchDescriptors(rec, d, ko[1:], ko[:-1])
        assert_same(a, b)
        assert_same(a, c)
        assert_same(a, mo.match_descriptors(to_records(d), d, ko[1:], ko[:-1]))
    finally:
        nd.close()


def test_device_variant_on_the_batch_result_leaves_it_unchanged(ob, synth, node):
    import torch
    pts, offs, rp = synth.generate(2, 40, scan_index_base=300)
    dev_pts = torch.from_numpy(pts).cuda()
    torch.cuda.synchronize()
    ko, K, p_kp, p_d = node.processBatchDevice(dev_pts.data_ptr(), offs, rp)
    assert K > 0
    # no synchronisation in between: the match is queued behind the batch on the context's stream
    m_dev = node.matchDescriptorsDevice(p_d, 1980, ko[1:], p_d, 1980, ko[:-1])
    kp_after = node.download(p_kp, (K, 4))
    d_after = node.download(p_d, (K, 1980))
    ko_h, kp_h, d_h = node.processBatch(pts, offs, rp)
    assert np.array_equal(ko, ko_h) and bits_equal(kp_after, kp_h) and bits_equal(d_after, d_h)
    m_host = node.matchDescriptors(d_h, d_h, ko[1:], ko[:-1])
    assert_same(m_dev, m_host)
    assert_same(m_dev, mo.match_descriptors(d_h, d_h, ko[1:], ko[:-1], n_threads=THREADS))
    # record output: the device pointer + 5 floats at stride 1996
    from feature_extraction_b200 import FeatureExtractionNode
    nd2 = FeatureExtractionNode(to_fe_params(ob.node_default()), max_points=8 << 20, max_scans=512, max_keypoints=1 << 15)
    try:
        nd2.enableRecordOutput(True)
        ko2, K2, p_kp2, p_rec = nd2.processBatchDevice(dev_pts.data_ptr(), offs, rp)
        rec_before = nd2.download(p_rec, (K2, 1996))
        m_rec = nd2.matchDescriptorsDevice(p_rec + 20, 1996, ko2[1:], p_rec + 20, 1996, ko2[:-1])
        assert_same(m_rec, m_dev)
        assert bits_equal(nd2.download(p_rec, (K2, 1996)), rec_before)
    finally:
        nd2.close()


def test_argument_errors_leave_the_context_usable(ob, synth, node):
    from feature_extraction_b200 import _native as N
    from feature_extraction_b200.node import FeatureExtractionError
    rng = np.random.default_rng(24)
    q = random_rows(rng, 6)
    r = random_rows(rng, 6)
    for bad in (dict(query_offsets=[0, 3, 2], ref_offsets=[0, 3, 6]),   # decreasing
                dict(query_offsets=[0, 3, 6], ref_offsets=[-1, 3, 6]),  # negative
                dict(query_offsets=[0, 7], ref_offsets=[0, 6])):        # beyond the rows passed
        with pytest.raises(ValueError):
            node.matchDescriptors(q, r, **bad)
    with pytest.raises(ValueError):
        node.matchDescriptorsDevice(1 << 20, 1979, [0, 1], 1 << 20, 1980, [0, 1])
    with pytest.raises(ValueError):
        node.matchDescriptorsDevice(0, 1980, [0, 1], 1 << 20, 1980, [0, 1])
    with pytest.raises(ValueError):
        node.matchDescriptors(q[:, :1000], r)
    # the raw C calls
    L = N.lib()
    res = N.MatchResult()
    qp, rp = q.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p)

    def call(f, qptr, qs, qo, rptr, rs, ro, G):
        qo = np.ascontiguousarray(qo, np.int64)
        ro = np.ascontiguousarray(ro, np.int64)
        return f(node._ctx, qptr, qs, qo.ctypes.data_as(C.c_void_p), rptr, rs, ro.ctypes.data_as(C.c_void_p), G, C.byref(res))

    for f in (L.fe_match_descriptors, L.fe_match_descriptors_device):
        assert call(f, qp, 1979, [0, 3], rp, 1980, [0, 3], 1) == N.FE_ERR_INVALID   # stride below 1980
        assert call(f, qp, 1980, [0, 3], rp, 1000, [0, 3], 1) == N.FE_ERR_INVALID
        assert call(f, qp, 1980, [0, 3, 2], rp, 1980, [0, 3, 6], 2) == N.FE_ERR_INVALID  # decreasing
        assert call(f, qp, 1980, [0, 3], rp, 1980, [-2, 3], 1) == N.FE_ERR_INVALID  # negative
        assert call(f, qp, 1980, [0, 3], rp, 1980, [0, 3], -1) == N.FE_ERR_INVALID  # n_groups < 0
        assert call(f, None, 1980, [0, 3], rp, 1980, [0, 3], 1) == N.FE_ERR_INVALID  # NULL with rows
        assert call(f, qp, 1980, [0, 3], None, 1980, [0, 3], 1) == N.FE_ERR_INVALID
        assert call(f, None, 1980, [2, 2], None, 1980, [0, 0], 1) == N.FE_OK  # no rows on either side
        assert call(f, qp, 1980, [0], rp, 1980, [0], 0) == N.FE_OK and res.n_queries == 0
    with pytest.raises(FeatureExtractionError):
        node._check(call(L.fe_match_descriptors, qp, 1979, [0, 3], rp, 1980, [0, 3], 1))
    # the context still matches and still runs batches correctly
    assert_same(node.matchDescriptors(q, r), mo.match_descriptors(q, r))
    P = ob.node_default()
    pts, offs, rpitch = synth.generate(2, 6, scan_index_base=77)
    ko, kp, d = node.processBatch(pts, offs, rpitch)
    ko_o, kp_o, d_o, _ = ob.process_batch(P, pts, offs, rpitch, mode=1, n_threads=THREADS)
    assert np.array_equal(ko, ko_o) and bits_equal(kp, kp_o) and bits_equal(d, d_o)
