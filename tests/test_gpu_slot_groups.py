"""The pipeline slots' arrays come in groups allocated once, in full, and freed only with the context (needs a B200).

A captured graph names the slot's arrays by address, so a group must never move; and a group the device cannot hold
must leave nothing half-built behind."""
import os

import numpy as np
import pytest

from match_cases import random_rows
from match_oracle import binding as mo
from util import bits_equal, check_descriptors, to_fe_params

pytestmark = pytest.mark.gpu


def test_replayed_graphs_survive_descriptors_over_a_wider_grid(ob, synth):
    """estimateDescriptors grids its own keypoints' bounding box.  Keypoints spread far wider than the crop box need
    the largest grid; the graphs captured before it still replay the oracle's bits afterwards."""
    from feature_extraction_b200 import FeatureExtractionNode
    P = ob.launch_playback()
    nd = FeatureExtractionNode(to_fe_params(P), max_points=1 << 18, max_scans=4, max_keypoints=1024)
    try:
        pts, offs, rp = synth.generate(1, 3, scan_index_base=9400)
        want = [ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1) for s in range(3)]
        assert all(len(w["keypoints"]) > 0 for w in want)
        one = np.array([0, 0], np.int64)

        def replay_all():
            for rep in range(3):           # eager, capture, replay
                for s in range(3):
                    sc = pts[offs[s]:offs[s + 1]]
                    one[1] = len(sc)
                    ko, kp, d = nd.processBatch(sc, one, rp[s:s + 1])
                    assert bits_equal(kp, want[s]["keypoints"]) and bits_equal(d, want[s]["descriptors"]), (rep, s)

        replay_all()
        replays = nd.enableGraphs(True)
        assert replays >= 3
        kps = want[0]["keypoints"].copy()
        far = np.array([[20.0, -300.0, 0.0, 0.0], [20.0, 300.0, 0.0, 0.0]], np.float32)
        kps = np.concatenate([kps, far])
        d_g = nd.estimateDescriptors(want[0]["cloud_full"], kps)
        d_o, _, _ = ob.estimate_descriptors(P, want[0]["cloud_full"], kps)
        assert check_descriptors(d_g, d_o)[1] == 0
        replay_all()
        assert nd.enableGraphs(True) >= replays + 9
    finally:
        nd.close()


def test_a_core_the_device_cannot_hold_is_refused_and_holds_nothing(ob):
    """With 2^26 keypoints per call the pipeline's core is more than 500 GB: its single allocation is refused, the
    staged points are never taken, every batch call says so, and calls that need no pipeline arrays still work."""
    from feature_extraction_b200 import FeatureExtractionNode, FeatureExtractionError, _native
    nd = FeatureExtractionNode(to_fe_params(ob.node_default()), max_keypoints=1 << 26)
    try:
        pts = np.zeros((100, 4), np.float32)
        pts[:, 0] = np.linspace(5.0, 20.0, 100)
        for _ in range(2):
            with pytest.raises(FeatureExtractionError) as e:
                nd.processBatch(pts, np.array([0, 100], np.int64), np.zeros((1, 2)))
            assert e.value.status == _native.FE_ERR_CUDA
        rng = np.random.default_rng(11)
        q, r = random_rows(rng, 40), random_rows(rng, 50)
        best, shift, d, sd = nd.matchDescriptors(q, r)
        o_best, o_shift, o_d, o_sd = mo.match_descriptors(q, r, n_threads=len(os.sched_getaffinity(0)))
        assert np.array_equal(best, o_best) and np.array_equal(shift, o_shift)
        assert bits_equal(d, o_d) and bits_equal(sd, o_sd)
    finally:
        nd.close()
