"""The CPU restatement of fe_loop_closures (match_oracle/fe_loop_oracle.cpp) against what the contract implies
(include/fe_b200.h, "loop closures"): constructed sequences, votes and candidate order from the matcher's output,
each candidate's verification from the matcher and registration directly, and the accuracy of the oracle chain on
out-and-back paths with ground truth (DESIGN.md §15)."""
import os
import re

import numpy as np
import pytest

from loop_cases import constructed, evaluate, oracle_chain
from match_oracle import binding as mo

THREADS = len(os.sched_getaffinity(0))


def defaults():
    from feature_extraction_b200 import loop_params_default
    p = loop_params_default()
    return p.min_gap, p.candidates


@pytest.mark.parametrize("case", range(6))
def test_constructed_sequences_give_what_the_contract_implies(case):
    kp, d, ko, so, cases, pole = constructed()
    c = cases[case]
    K = c["candidates"]
    o = mo.loop_closures(kp, d, ko, so, c["min_gap"], K)
    for s, w in c["want"].items():
        for k, v in w.items():
            assert o[k][s].tolist() == v, (case, s, k, o[k][s], v)
    first = np.repeat(so[:-1], np.diff(so))
    for s in range(len(ko) - 1):
        a = o["assoc"][ko[s] - ko[0]:ko[s + 1] - ko[0]]
        if s - first[s] < c["min_gap"]:  # not eligible
            assert o["loop"][s] == -1 and (o["cand_scan"][s] == -1).all() and (o["cand_status"][s] == -1).all()
        if o["loop"][s] < 0:
            assert (a == -1).all() and o["loop_scan"][s] == -1 and o["n_inliers"][s] == 0
            assert (o["pose"][s] == [1.0, 0.0, 0.0, 0.0]).all()
            continue
        # every inlier is a row of the loop scan at the same pole; the winner's outputs are its candidate's
        j, k = o["loop_scan"][s], o["loop"][s]
        inl = a >= 0
        assert ((a[inl] >= ko[j]) & (a[inl] < ko[j + 1])).all()
        assert (pole[a[inl]] == pole[ko[s]:ko[s + 1]][inl]).all(), s
        assert inl.sum() == o["n_inliers"][s] == o["cand_inliers"][s, k]
        assert o["cand_scan"][s, k] == j and o["cand_status"][s, k] == 2
        assert np.array_equal(o["pose"][s].view(np.uint64), o["cand_pose"][s, k].view(np.uint64))
    # scans without a candidate at a rank: votes 0, status -1, identity pose
    none = o["cand_scan"] == -1
    assert (o["cand_votes"][none] == 0).all() and (o["cand_status"][none] == -1).all()
    assert (o["cand_pose"][none] == [1.0, 0.0, 0.0, 0.0]).all()


def _votes(best, ko, s, first):
    """The contract's votes from the matcher's `best` over scan s's database: [(scan, votes)] in candidate order."""
    v = {}
    for b in best:
        if b >= 0:
            j = int(np.searchsorted(ko[first:], b, side="right")) - 1 + first
            assert ko[j] <= b < ko[j + 1]
            v[j] = v.get(j, 0) + 1
    return sorted(v.items(), key=lambda x: (-x[1], x[0]))


def _check_against_parts(kp, d, ko, so, gap, K, o, **reg):
    first = np.repeat(so[:-1], np.diff(so))
    for s in range(len(ko) - 1):
        f = first[s]
        if s - f < gap or ko[s + 1] == ko[s]:
            assert (o["cand_scan"][s] == -1).all()
            continue
        best = mo.match_descriptors(d, d, [ko[s], ko[s + 1]], [ko[f], ko[s - gap + 1]], n_threads=THREADS)[0]
        want = _votes(best, ko, s, f)[:K]
        got = [(int(j), int(v)) for j, v in zip(o["cand_scan"][s], o["cand_votes"][s]) if j >= 0]
        assert got == want, (s, got, want)
        for k, (j, _) in enumerate(want):
            b2 = mo.match_descriptors(d, d, [ko[s], ko[s + 1]], [ko[j], ko[j + 1]])[0]
            r = mo.register_matches(kp, kp, b2, [ko[s], ko[s + 1]], [ko[j], ko[j + 1]], **reg)
            for key in ("status", "n_inliers", "n_hypotheses"):
                assert o["cand_" + key.replace("n_", "")][s, k] == r[key][0], (s, k, key)
            assert o["cand_rms"][s, k].view(np.uint64) == r["rms"][0].view(np.uint64)
            assert np.array_equal(o["cand_pose"][s, k].view(np.uint64), r["pose"][0].view(np.uint64))
            if o["loop"][s] == k:
                assert np.array_equal(o["assoc"][ko[s] - ko[0]:ko[s + 1] - ko[0]], r["assoc"])


def test_votes_candidates_and_verification_are_the_matcher_and_registration_s():
    kp, d, ko, so, cases, _ = constructed()
    for c in cases:
        o = mo.loop_closures(kp, d, ko, so, c["min_gap"], c["candidates"])
        _check_against_parts(kp, d, ko, so, c["min_gap"], c["candidates"], o)
    ko4, kp4, d4, _ = oracle_chain(4, "loop", 0)
    so4 = np.array([0, len(ko4) - 1])
    for gap, K, reg in ((5, 4, {}), (10, 2, dict(min_inliers=8))):
        o = mo.loop_closures(kp4, d4, ko4, so4, gap, K, n_threads=THREADS, **reg)
        assert (o["loop"] >= 0).sum() >= 5
        _check_against_parts(kp4, d4, ko4, so4, gap, K, o, **reg)


def test_defaults_are_the_header_s():
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "fe_b200.h")).read()
    gap = int(re.search(r"#define FE_LOOP_MIN_GAP_DEFAULT (\d+)", header).group(1))
    K = int(re.search(r"#define FE_LOOP_CANDIDATES_DEFAULT (\d+)", header).group(1))
    assert defaults() == (gap, K)


def test_invalid_arguments():
    kp, d, ko, so, _, _ = constructed()
    mo.loop_closures(kp, d, ko, so, 1, 1)
    for gap, K, kw in ((0, 1, {}), (1, 0, {}), (1, 17, {}), (1, 1, dict(min_inliers=0)), (1, 1, dict(inlier_radius=-1.0))):
        with pytest.raises(ValueError):
            mo.loop_closures(kp, d, ko, so, gap, K, **kw)
    with pytest.raises(ValueError):
        mo.loop_closures(kp, d, ko, so[:-1], 1, 1)  # does not end at B
    empty = mo.loop_closures(kp[:0], d[:0], [0], [0], 1, 2)
    assert all(len(v) == 0 for v in empty.values())
    one = mo.loop_closures(kp[:0], d[:0], [0, 0], [0, 0, 1, 1], 1, 2)
    assert list(one["loop"]) == [-1] and one["cand_scan"].tolist() == [[-1, -1]]


# Accuracy of the oracle chain at the defaults (DESIGN.md §15): a floor a little under the measured found fraction of
# config 4, and no wrong loop in either configuration, out-and-back or forward.
FLOOR = 0.82


@pytest.mark.parametrize("cfg", [2, 4])
def test_sequence_evaluation(cfg):
    gap, K = defaults()
    r = evaluate(cfg, gap, K, threads=THREADS)
    print("config %d min_gap %d candidates %d: %d revisits, found %.3f, wrong %d" % (cfg, gap, K, r["revisits"],
                                                                                   r["fraction"], r["wrong"]))
    assert r["wrong"] == 0
    if cfg == 4:
        assert r["fraction"] >= FLOOR
        # against odometry's own relative pose of the same pairs, the loops are far closer to the truth
        assert np.median(r["dt"]) < np.median(r["odo_dt"]) and max(r["dt"]) < 0.5
    else:
        assert r["found"] == 0  # about 3 keypoints a scan: never 16 inliers
