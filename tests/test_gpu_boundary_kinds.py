"""The tolerance-boundary report over all ten kinds on the device (fe_enable_boundary_report_all) against the CPU
oracle's counts (boundary_oracle/), element for element, through every batch route; the report changes no result."""
import numpy as np
import pytest

import boundary_cases as bc
from boundary_oracle import binding as bo
from util import bits_equal, to_fe_params

pytestmark = pytest.mark.gpu


def _params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


def _node(P, max_scans=64):
    from feature_extraction_b200 import FeatureExtractionNode
    return FeatureExtractionNode(to_fe_params(P), max_points=1 << 22, max_scans=max_scans, max_keypoints=1 << 14)


@pytest.mark.parametrize("cfg,nscans", [(1, 4), (2, 32), (3, 2), (4, 3)])
def test_all_kinds_equal_the_oracles_on_every_route(ob, synth, cfg, nscans):
    import torch
    P = _params(ob, cfg)
    pts, offs, rp = synth.generate(cfg, nscans, scan_index_base=41200)
    nd = _node(P)
    ko0, kp0, d0 = nd.processBatch(pts, offs, rp)
    for eps in (1e-6, 1e-4):
        want = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=eps, mode=1, n_threads=8)
        nd.enableBoundaryReport(eps)
        ko1, kp1, d1 = nd.processBatch(pts, offs, rp)
        rep4 = nd.boundaryReport()
        with pytest.raises(Exception):
            nd.boundaryReportAll()          # enabled for the radius kinds only
        nd.enableBoundaryReportAll(eps)
        ko, kp, d = nd.processBatch(pts, offs, rp)
        rep = nd.boundaryReportAll()
        assert rep.shape == (nscans, 10)
        assert np.array_equal(rep, want), (eps, rep.sum(0), want.sum(0))
        assert np.array_equal(nd.boundaryReport(), rep[:, :4]) and np.array_equal(rep4, rep[:, :4])
        for o, k, dd in ((ko1, kp1, d1), (ko, kp, d)):
            assert np.array_equal(o, ko0) and bits_equal(k, kp0) and bits_equal(dd, d0)
        # several sub-batches on both slots
        small = _node(P, max_scans=max(1, nscans // 3))
        small.enableBoundaryReportAll(eps)
        small.processBatch(pts, offs, rp)
        assert np.array_equal(small.boundaryReportAll(), want)
        small.close()
        # device-resident input
        dev = torch.from_numpy(pts).cuda()
        torch.cuda.synchronize()
        nd.processBatchDevice(dev.data_ptr(), offs, rp)
        assert np.array_equal(nd.boundaryReportAll(), want)
        # 32-byte records decoded on the device
        raw = np.zeros((len(pts), 8), np.float32)
        raw[:, :4] = pts
        nd.processBatchLayout(raw.view(np.uint8), 32, 0, 4, 8, offs, rp)
        assert np.array_equal(nd.boundaryReportAll(), want)
        # K2 through the grid-based kernels only
        nd.forceGridClustering(True)
        nd.processBatch(pts, offs, rp)
        assert np.array_equal(nd.boundaryReportAll(), want)
        nd.forceGridClustering(False)
    nd.close()


@pytest.mark.parametrize("cfg", [2, 4])
def test_graph_replay_and_lean_rerun_count_once(ob, synth, cfg):
    P = _params(ob, cfg)
    pts, offs, rp = synth.generate(cfg, 3, scan_index_base=41900)
    want = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=1e-4, mode=1, n_threads=8)
    nd = _node(P, max_scans=16)
    nd.enableBoundaryReportAll(1e-4)
    r0 = nd.leanReruns()
    for rep in range(3):                    # eager, capture, replay
        nd.processBatch(pts, offs, rp)
        assert np.array_equal(nd.boundaryReportAll(), want), rep
    if cfg == 4:                            # K4d's larger instantiations: the lean chain was run again
        assert nd.leanReruns() > r0
    nd.close()


def test_switching_between_radius_and_all_kinds_never_replays_a_stale_graph(ob, synth):
    P = _params(ob, 2)
    pts, offs, rp = synth.generate(2, 4, scan_index_base=42100)
    want = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=1e-4, mode=1, n_threads=8)
    nd = _node(P, max_scans=16)
    for rep in range(2):
        for all_kinds in (False, True, False):
            for _ in range(3):
                if all_kinds:
                    nd.enableBoundaryReportAll(1e-4)
                else:
                    nd.enableBoundaryReport(1e-4)
                nd.processBatch(pts, offs, rp)
                assert np.array_equal(nd.boundaryReport(), want[:, :4])
                if all_kinds:
                    assert np.array_equal(nd.boundaryReportAll(), want)
                else:
                    with pytest.raises(Exception):
                        nd.boundaryReportAll()
    nd.close()


def test_without_descriptors_the_3dsc_kinds_are_zero(ob, synth):
    P = _params(ob, 2)
    P.estimate_descriptors = 0
    pts, offs, rp = synth.generate(2, 8, scan_index_base=42300)
    want = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=1e-2, mode=1, n_threads=8)
    nd = _node(P)
    nd.enableBoundaryReportAll(1e-2)
    nd.processBatch(pts, offs, rp)
    rep = nd.boundaryReportAll()
    assert np.array_equal(rep, want) and not rep[:, 7:].any() and rep[:, 4:7].any()
    nd.close()


@pytest.mark.parametrize("kind", [4, 5, 6, 7, 8, 9])
def test_constructed_decisions_count_as_on_the_cpu(ob, kind):
    for off in (bc.NEAR, -bc.NEAR, bc.FAR, 0.0):
        if off == 0.0 and kind != 9:
            continue
        P, pts, offs, rp = bc.case(ob, kind, off)
        want = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=bc.EPS, mode=0)
        nd = _node(P, max_scans=4)
        nd.enableBoundaryReportAll(bc.EPS)
        nd.processBatch(pts, offs, rp)
        assert np.array_equal(nd.boundaryReportAll(), want), (kind, off)
        nd.close()
