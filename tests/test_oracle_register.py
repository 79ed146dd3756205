"""The CPU restatement of fe_register_matches (match_oracle/fe_register_oracle.cpp) against what the contract implies
(include/fe_b200.h, "registration"), an independent numpy evaluation, and the accuracy of the whole chain (oracle
pipeline, oracle matcher, oracle registration) on synthetic scan sequences with ground truth."""
import numpy as np
import pytest

from match_oracle import binding as mo
from register_cases import PARAMS, apply, constructed, errors, hypothesis_pairs, oracle_params, relative, sequence

DEFAULT = dict(inlier_radius=0.5, min_separation=1.0, max_hypotheses=512, min_inliers=16, refine_iterations=4)


def test_constructed_cases_give_what_the_contract_implies():
    q, r, best, qo, ro, want = constructed()
    o = mo.register_matches(q, r, best, qo, ro, **PARAMS)
    for g, w in enumerate(want):
        for k in ("status", "n_inliers", "n_hypotheses"):
            if k in w:
                assert o[k][g] == w[k], (g, k, o[k][g], w[k])
        if "pose" in w:
            assert np.abs(o["pose"][g] - w["pose"]).max() < 1e-9, (g, o["pose"][g], w["pose"])
        a = o["assoc"][qo[g] - qo[0]:qo[g + 1] - qo[0]]
        if "assoc_of" in w:
            assert list(a) == [-1 if j < 0 else ro[g] + j for j in w["assoc_of"]], (g, a)
        if w["status"] == 0:
            assert list(o["pose"][g]) == [1.0, 0.0, 0.0, 0.0] and o["rms"][g] == 0.0 and o["n_inliers"][g] == 0
            assert (a == -1).all()
    # rows outside every group are not touched, and n_groups = 0 gives empty results
    empty = mo.register_matches(q, r, best[:0], qo[:1], ro[:1])
    assert all(len(v) == 0 for v in empty.values())


def test_the_hypothesis_map_visits_every_pair_or_evenly_spaced_ones():
    for n_c in (2, 3, 10, 33, 40, 200):
        P = n_c * (n_c - 1) // 2
        for H in (1, 7, 512, 65536):
            idx = hypothesis_pairs(n_c, H)
            assert len(idx) == min(P, H) and len(set(idx)) == len(idx) and idx[0] == 0
            if P <= H:
                assert idx == list(range(P))
            else:
                assert set(np.diff(idx)) <= {P // H, -(-P // H)}


@pytest.mark.parametrize("max_hypotheses", [1, 50, 779, 780, 1000])
def test_hypothesis_count_follows_the_map(max_hypotheses):
    """40 correspondences; row 0 is matched to the wrong reference row, so that the pairs (0, b) whose length changes by
    2 * radius or more are rejected.  The oracle's count must equal a numpy restatement over the map's pairs."""
    g40 = np.array([[5.0 * a, 7.0 * b] for a in range(8) for b in range(5)])
    from register_cases import kp
    q, r = kp(g40), kp(g40 + [1.0, 2.0])
    best = np.arange(40)
    best[0] = 39
    o = mo.register_matches(q, r, best, [0, 40], [0, 40], max_hypotheses=max_hypotheses, min_inliers=3)
    pairs = [(a, b) for a in range(40) for b in range(a + 1, 40)]
    pq, pr = q[:, :2].astype(np.float64), r[:, :2].astype(np.float64)
    n = 0
    for i in hypothesis_pairs(40, max_hypotheses):
        a, b = pairs[i]
        lu = np.sum((pq[b] - pq[a]) ** 2)
        lv = np.sum((pr[best[b]] - pr[best[a]]) ** 2)
        n += lu >= 1.0 and lv >= 1.0 and abs(np.sqrt(lu) - np.sqrt(lv)) < 1.0
    assert o["n_hypotheses"][0] == n
    if n == 0:  # max_hypotheses = 1: pair (0, 1) only, which contains the wrong match
        assert o["status"][0] == 0
    else:
        assert o["status"][0] == 2 and o["n_inliers"][0] == 40


def least_squares(qxy, rxy):
    """Planar rigid least squares of rxy ~ R qxy + t (numpy, float64, its own summation order)."""
    mp, mq = qxy.mean(axis=0), rxy.mean(axis=0)
    a, b = qxy - mp, rxy - mq
    A = np.sum(a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1])
    B = np.sum(a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0])
    n = np.hypot(A, B)
    c, s = A / n, B / n
    return np.array([c, s, mq[0] - (c * mp[0] - s * mp[1]), mq[1] - (s * mp[0] + c * mp[1])])


def test_refined_motion_is_the_least_squares_fit_of_its_inliers(ob, synth):
    """With enough rounds the refinement converges: the final motion is the least-squares fit of its own inliers."""
    pts, offs, rp, poses = sequence(synth, 4, 0)
    ko, kp, d, _ = ob.process_batch(oracle_params(ob, 4), pts, offs, rp, mode=0, n_threads=8)
    best = mo.match_descriptors(d, d, ko[1:], ko[:-1], n_threads=8)[0]
    o = mo.register_matches(kp, kp, best, ko[1:], ko[:-1], refine_iterations=100, min_inliers=3)
    checked = 0
    for g in np.nonzero(o["n_inliers"] >= 2)[0]:
        rows = np.arange(ko[g + 1], ko[g + 2])
        a = o["assoc"][rows - ko[1]]
        inl = a >= 0
        ls = least_squares(kp[rows[inl], :2].astype(np.float64), kp[a[inl], :2].astype(np.float64))
        assert np.abs(ls - o["pose"][g]).max() < 1e-9, (g, ls, o["pose"][g])
        w = apply(o["pose"][g], kp[rows, :2])
        d2 = np.sum((w[inl] - kp[a[inl], :2].astype(np.float64)) ** 2, axis=1)
        assert abs(np.sqrt(d2.mean()) - o["rms"][g]) < 1e-9
        checked += 1
    assert checked >= 15


# Accuracy of the chain on 20 sequences of 20 scans per configuration (DESIGN.md §13).  With the default parameters no
# registered pair may be off by more than 0.5 m or 2 deg; the floor of the registered fraction sits a little under the
# measured one.
FLOOR = {2: 0.0, 4: 0.70}


@pytest.mark.parametrize("cfg", [2, 4])
def test_sequence_evaluation(ob, synth, cfg):
    st, dts, dys = [], [], []
    for seq in range(20):
        pts, offs, rp, poses = sequence(synth, cfg, seq)
        ko, kp, d, _ = ob.process_batch(oracle_params(ob, cfg), pts, offs, rp, mode=0, n_threads=8)
        best = mo.match_descriptors(d, d, ko[1:], ko[:-1], n_threads=8)[0]
        o = mo.register_matches(kp, kp, best, ko[1:], ko[:-1], **DEFAULT)
        dt, dyaw = errors(o["pose"], relative(poses))
        st.append(o["status"])
        dts.append(dt)
        dys.append(np.degrees(dyaw))
    st, dt, dy = np.concatenate(st), np.concatenate(dts), np.concatenate(dys)
    ok = st == 2
    print("config %d: %d pairs, registered %.3f; translation error median %.4f max %.4f m, yaw error median %.4f max %.4f deg"
          % (cfg, len(st), ok.mean(), np.median(dt[ok]) if ok.any() else np.nan, dt[ok].max() if ok.any() else np.nan,
             np.median(dy[ok]) if ok.any() else np.nan, dy[ok].max() if ok.any() else np.nan))
    assert ok.mean() >= FLOOR[cfg]
    assert not ((dt[ok] > 0.5) | (dy[ok] > 2.0)).any()
