"""The CPU oracle's tolerance-boundary report over all ten kinds (boundary_oracle/, fe_enable_boundary_report_all):
consistent with the four-kind report, independent of the search back end, monotone in eps, and counting exactly
the constructed decisions of tests/boundary_cases.py — which do flip when moved by 2 eps across their boundary."""
import numpy as np
import pytest

import boundary_cases as bc
from boundary_oracle import binding as bo


def _cfg_params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


@pytest.mark.parametrize("cfg", [2, 4])
def test_all_kinds_extend_the_radius_report(ob, synth, cfg):
    P = _cfg_params(ob, cfg)
    pts, offs, rp = synth.generate(cfg, 6 if cfg == 2 else 3, scan_index_base=31000)
    prev = None
    for eps in (1e-6, 1e-4, 1e-2):
        rep = bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=eps, mode=1, n_threads=4)
        assert rep.shape == (len(offs) - 1, 10) and rep.dtype == np.int64
        assert np.array_equal(rep[:, :4], ob.process_batch_boundary(P, pts, offs, rp, eps_m=eps, mode=1, n_threads=4))
        assert np.array_equal(rep, bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=eps, mode=0, n_threads=4))
        if prev is not None:
            assert (rep >= prev).all(), "a count fell as eps grew"
        if eps == 1e-4:
            assert rep[:, 4:].sum() > 0, "no new kind met at 1e-4 m"
        prev = rep


def _counts(ob, kind, offset):
    P, pts, offs, rp = bc.case(ob, kind, offset)
    return bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=bc.EPS, mode=0)[0]


def _base(ob, kind):
    P, pts, offs, rp = bc.base_case(ob, kind)
    if len(pts) == 0:
        return np.zeros(10, np.int64)
    return bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=bc.EPS, mode=0)[0]


@pytest.mark.parametrize("kind", [4, 5, 6, 7, 8, 9])
def test_constructed_decision_is_counted_near_and_not_far(ob, kind):
    base = _base(ob, kind)
    for off in (bc.NEAR, -bc.NEAR):
        assert _counts(ob, kind, off)[kind] == base[kind] + 1, off
    assert _counts(ob, kind, bc.FAR)[kind] == base[kind]


def test_crop_point_far_outside_on_another_axis_is_not_counted(ob):
    P = bc.params(ob)
    pts, offs, rp = bc._scan([bc.crop_point(bc.NEAR, x=P.x_max + 1.0)])
    assert bo.process_batch_boundary_all(P, pts, offs, rp, eps_m=bc.EPS, mode=0)[0][4] == 0


def test_neighbour_straight_above_the_keypoint_is_an_azimuth_boundary(ob):
    assert _counts(ob, 9, 0.0)[9] == _base(ob, 9)[9] + 1


def test_moving_by_two_eps_flips_the_decision(ob):
    shift = bc.NEAR - 2 * bc.EPS
    P = bc.params(ob)
    # [4] the crop keeps the point only on the inner side
    a, b = (ob.filter_cloud(P, bc._scan([bc.crop_point(o)])[0]) for o in (bc.NEAR, shift))
    assert (len(a), len(b)) == (0, 1)
    # [5] ring membership: window [2, 4] (ring 9) on one side, [0, 2] (ring 8) on the other
    for off, ring in ((bc.NEAR, 9), (shift, 8)):
        c = ob.get_elevation_angles(bc._scan([bc.ring_point(off / (bc.RANGE * bc.DEG))])[0])
        assert len(ob.select_ring(c, ring)) == 1 and len(ob.select_ring(c, 17 - ring)) == 0
    # [6] the gate passes the cluster only below 2 x threshold: one keypoint more
    n = [len(ob.get_cylinder_segments(P, ob.get_elevation_angles(bc._scan(bc.cluster(0.3 + o))[0]))[0]) for o in (bc.NEAR, shift)]
    assert n == [0, 1]
    # [7], [8] the neighbour's contribution lands in another descriptor bin
    for kind in (7, 8):
        d = []
        for off in (bc.NEAR, shift):
            Pd, pts, offs, rp = bc.case(ob, kind, off)
            d.append(ob.process_batch(Pd, pts, offs, rp, mode=0)[2])
        assert d[0].shape == d[1].shape == (1, 1980)
        assert not np.array_equal(d[0] != 0, d[1] != 0), kind
