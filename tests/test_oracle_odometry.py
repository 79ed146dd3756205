"""The CPU restatement of fe_odometry (match_oracle/fe_odometry_oracle.cpp) against what the contract implies
(include/fe_b200.h, "odometry"): constructed sequences, the pose chain, W = 1 against the registration oracle, and the
accuracy of the oracle chain on synthetic scan sequences with ground truth (DESIGN.md §14)."""
import os
import re

import numpy as np
import pytest

from match_oracle import binding as mo
from odometry_cases import IDENTITY, chain, constructed, evaluate, oracle_chain, scan_pairs_best
from feature_extraction_b200 import ODOMETRY_WINDOW as DEFAULT_WINDOW
from register_cases import kp as make_kp


@pytest.mark.parametrize("W", [1, 2, 4, 64])
def test_constructed_sequences_give_what_the_contract_implies(W):
    kp, ko, best, so, seqs, pole = constructed()
    o = mo.odometry(kp, ko, best, so, W)
    for q in seqs:
        for s, w in q["want"](W).items():
            for k, v in w.items():
                assert o[k][q["scans"] + s] == v, (W, q["scans"], s, k, o[k][q["scans"] + s], v)
    first = np.zeros(len(ko) - 1, bool)
    first[so[:-1][np.diff(so) > 0]] = True
    assert (o["source"][first] == 0).all() and (o["status"][first] == -1).all()
    assert (o["motion"][first] == IDENTITY).all() and (o["pose"][first] == IDENTITY).all()
    assert (o["n_inliers"][first] == 0).all() and (o["rms"][first] == 0).all()
    for f in np.nonzero(first)[0]:
        assert (o["assoc"][ko[f] - ko[0]:ko[f + 1] - ko[0]] == -1).all()
    # a predicted link is the previous motion (constant velocity), or the identity at t = 1
    for s in np.nonzero(o["source"] == 2)[0]:
        want = IDENTITY if o["source"][s - 1] == 0 else o["motion"][s - 1]
        assert np.array_equal(o["motion"][s].view(np.uint64), want.view(np.uint64)), s
    assert np.array_equal(o["motion"][5], o["motion"][4])  # sequence 1, link 2 repeats link 1
    # every inlier lies in its window: scan t-1 or an earlier scan of the sequence, and holds the same pole
    for s in range(len(ko) - 1):
        a = o["assoc"][ko[s] - ko[0]:ko[s + 1] - ko[0]]
        inl = a >= 0
        assert (pole[a[inl]] == pole[ko[s]:ko[s + 1]][inl]).all(), s
        assert inl.sum() == o["n_inliers"][s] or o["source"][s] == 0
    # sequence 0, W >= 2: pole 16 of scan 2 is an inlier of scan 0's row of it
    row16 = ko[2] + 15
    assert pole[row16] == 16
    assert o["assoc"][row16] == (ko[0] + 16 if W >= 2 else -1)
    # sequence 1: the predicted link 2 cuts the window of link 3, whose pole-16 row stays without an inlier
    assert o["assoc"][ko[7] - 1] == -1 and pole[ko[7] - 1] == 16


def test_the_cut_window_would_have_seen_more():
    """Sequence 1's link 3 against scans 1 and 2, placed by the true motions, scores 17: so the 16 of the odometry are
    the cut window's, not a coincidence of the scene."""
    kp, ko, best, so, seqs, pole = constructed()
    o = mo.odometry(kp, ko, best, so, 1)
    m2 = o["motion"][5]
    inv2 = np.array([m2[0], -m2[1], -(m2[0] * m2[2] + m2[1] * m2[3]), m2[1] * m2[2] - m2[0] * m2[3]])
    s1 = kp[ko[4]:ko[5]].astype(np.float64)
    placed = np.stack([inv2[0] * s1[:, 0] - inv2[1] * s1[:, 1] + inv2[2], inv2[1] * s1[:, 0] + inv2[0] * s1[:, 1] + inv2[3]], 1)
    ref = np.concatenate([make_kp(placed), kp[ko[5]:ko[6]]])
    b = best[ko[6] - ko[1]:ko[7] - ko[1]]
    b = np.where(b < 0, -1, b - ko[5] + len(s1))
    r = mo.register_matches(kp[ko[6]:ko[7]], ref, b, [0, ko[7] - ko[6]], [0, len(ref)])
    assert r["n_inliers"][0] == 17 and o["n_inliers"][6] == 16


@pytest.mark.parametrize("W", [1, 3])
def test_poses_are_the_composed_motions(W):
    kp, ko, best, so, _, _ = constructed()
    o = mo.odometry(kp, ko, best, so, W)
    assert np.array_equal(chain(o["motion"], o["source"]).view(np.uint64), o["pose"].view(np.uint64))
    ko4, kp4, best4, _ = oracle_chain(4, 0)
    o = mo.odometry(kp4, ko4, best4, [0, len(ko4) - 1], W)
    assert np.array_equal(chain(o["motion"], o["source"]).view(np.uint64), o["pose"].view(np.uint64))


def _same_as_pairs(o, reg, ko, so):
    first = set(np.asarray(so)[:-1].tolist())
    for s in range(1, len(ko) - 1):
        if s in first:
            continue
        g = s - 1
        for k in ("status", "n_inliers", "n_hypotheses"):
            assert o[k][s] == reg[k][g], (s, k)
        assert o["rms"][s].view(np.uint64) == reg["rms"][g].view(np.uint64), s
        if reg["status"][g] == 2:
            assert np.array_equal(o["motion"][s].view(np.uint64), reg["pose"][g].view(np.uint64)), s
        assert np.array_equal(o["assoc"][ko[s] - ko[0]:ko[s + 1] - ko[0]], reg["assoc"][ko[s] - ko[1]:ko[s + 1] - ko[1]]), s


def test_window_one_is_registration_of_each_scan_against_the_previous():
    kp, ko, best, so, _, _ = constructed()
    reg = mo.register_matches(kp, kp, scan_pairs_best(ko, best, so), ko[1:], ko[:-1])
    _same_as_pairs(mo.odometry(kp, ko, best, so, 1), reg, ko, so)
    for cfg in (2, 4):
        ko_, kp_, best_, _ = oracle_chain(cfg, 1)
        for kw in ({}, dict(min_inliers=3)):
            reg = mo.register_matches(kp_, kp_, best_, ko_[1:], ko_[:-1], **kw)
            _same_as_pairs(mo.odometry(kp_, ko_, best_, [0, len(ko_) - 1], 1, **kw), reg, ko_, [0, len(ko_) - 1])


def test_default_window_is_the_header_s():
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "fe_b200.h")).read()
    assert int(re.search(r"#define FE_ODOMETRY_WINDOW_DEFAULT (\d+)", header).group(1)) == DEFAULT_WINDOW


def test_invalid_arguments():
    kp, ko, best, so, _, _ = constructed()
    mo.odometry(kp, ko, best, so, 1)
    for bad in (dict(window=0), dict(window=65), dict(min_inliers=0), dict(inlier_radius=-1.0)):
        with pytest.raises(ValueError):
            mo.odometry(kp, ko, best, so, **{"window": 1, **bad})
    with pytest.raises(ValueError):
        mo.odometry(kp, ko, best, so[:-1], 1)  # does not end at B
    wrong = best.copy()
    wrong[ko[2] - ko[1]] = ko[0]  # scan 2's row into scan 0: not the previous scan
    with pytest.raises(ValueError):
        mo.odometry(kp, ko, wrong, so, 2)
    empty = mo.odometry(kp[:0], [0], np.zeros(0, np.int64), [0], 1)
    assert all(len(v) == 0 for v in empty.values())
    one = mo.odometry(kp[:0], [0, 0], np.zeros(0, np.int64), [0, 0, 1, 1], 1)
    assert list(one["source"]) == [0] and list(one["status"]) == [-1]


# Accuracy of the oracle chain (DESIGN.md §14): floors of the registered fraction a little under the measured values,
# and no wrong link at the default window.
FLOOR = {(4, 1): 0.75, (4, 2): 0.80, (4, 4): 0.80, (4, 8): 0.80}


@pytest.mark.parametrize("cfg", [2, 4])
def test_sequence_evaluation(cfg):
    rows = {}
    for W in (1, 2, 4, 8):
        frac, wrong, dt, dy = evaluate(cfg, W)
        rows[W] = (frac, wrong)
        print("config %d W %d: registered %.3f, wrong %d; end point %.3f / %.3f m, %.3f / %.3f deg (median / max)"
              % (cfg, W, frac, wrong, np.median(dt), dt.max(), np.median(dy), dy.max()))
        if cfg == 4:
            assert frac >= FLOOR[(cfg, W)], (W, frac)
        else:
            assert frac == 0.0  # about 3 keypoints a scan: never 16 inliers
    assert rows[DEFAULT_WINDOW][1] == 0
    if cfg == 4:
        assert abs(rows[1][0] - 0.758) < 0.0015 and rows[1][1] == 0  # W = 1 is scan against scan (DESIGN.md §13)
