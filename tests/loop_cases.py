"""Inputs of the loop-closure tests (include/fe_b200.h, "loop closures"): constructed sequences whose votes, candidates
and loops are known exactly, out-and-back paths that revisit their own start, and the oracle chain with its evaluation
against the ground truth (DESIGN.md §15)."""
import functools

import numpy as np

from odometry_cases import POLES, _in_frame
from register_cases import C24, S7, errors, kp, oracle_params, sequence

DESC = 1980


# ---- constructed sequences ------------------------------------------------------------------------------------------

NODESC, MOVED = 100, 200  # a pole index + NODESC: the pole's position without a descriptor; + MOVED: its descriptor, moved


def pole_rows(poles):
    """One descriptor row per pole, identical wherever that pole appears: row p is 1 at bin p of every azimuth block, 0
    elsewhere, so every shift gives the same distance: 0 between two rows of one pole, 24 between two poles.  A row
    with NODESC is all NaN (no neighbours): it never matches and is never matched."""
    d = np.zeros((len(poles), DESC), np.float32)
    for i, p in enumerate(poles):
        if p >= NODESC and p < MOVED:
            d[i] = np.nan
        else:
            d[i, p % 100 + 165 * np.arange(12)] = 1.0
    return d


def constructed():
    """Sequences with known loop closures under the default registration parameters (min_inliers = 16).
    -> kp, descriptors, keypoint_offsets, sequence_offsets, cases, pole.  Each case is a dict of the sequence's first
    absolute scan (`scans`), the min_gap and candidates it is meant for, and `want` = {absolute scan: {field: value}}
    (cand_* fields as lists over the ranks).  pole: absolute row -> the pole at that row's position (-1: a row far
    from every pole)."""
    rows, desc, pole, ko, so = [], [], [], [0], [0]
    R = lambda *a: list(range(*a))  # noqa: E731
    mv = lambda tx, ty: np.array([1.0, 0.0, tx, ty])  # noqa: E731
    ident = np.array([1.0, 0.0, 0.0, 0.0])

    def seq(frames, visible):
        """visible[t]: per row a pole index, + NODESC or + MOVED (scaled by 1.37 about the origin, so that no rigid
        motion maps it back), or -1 (no descriptor, far from every pole)."""
        s0 = len(ko) - 1
        for frame, vis in zip(frames, visible):
            xy = np.full((len(vis), 2), 900.0)
            for i, p in enumerate(vis):
                if p >= 0:
                    xy[i] = _in_frame(frame, POLES[[p % 100]] * (1.37 if p >= MOVED else 1.0))[0]
            rows.append(kp(xy))
            desc.extend(NODESC if p < 0 else p for p in vis)
            pole.extend(-1 if p < 0 or p >= MOVED else p % 100 for p in vis)
            ko.append(ko[-1] + len(vis))
        so.append(len(ko) - 1)
        return s0

    cases = []
    # 0: scan 3 revisits scan 0 (18 poles), turned and moved; scans 1 and 2 hold other poles and pole 0.  min_gap 2:
    #    scan 2's database is scan 0, where its 8 rows all find a best (distinct poles are 24 apart, not NaN): 8 votes,
    #    and every match lands on scan 0's first row, so every pair is rejected.  Scan 3's poles 0-17 vote for scan 0,
    #    18 and 19 for scan 1; scan 0 registers with 18 inliers, scan 1 with 3 (poles 0, 18, 19).
    s = seq([ident, mv(2, 0), mv(4, 0), np.array([C24, S7, 25.0, -25.0])],
            [R(18), R(18, 23) + [0], R(18, 25) + [0], R(18) + [18, 19]])
    cases.append({"scans": s, "min_gap": 2, "candidates": 2, "want": {
        s + 2: {"loop": -1, "cand_scan": [s, -1], "cand_votes": [8, 0], "cand_status": [0, -1], "cand_hypotheses": [0, 0]},
        s + 3: {"loop": 0, "loop_scan": s, "n_inliers": 18, "cand_scan": [s, s + 1], "cand_votes": [18, 2],
                "cand_inliers": [18, 3], "cand_status": [2, 1]}}})
    # 1: a tie in votes broken by scan index: scan 2's poles 0-11 find their descriptors only in scan 0, poles 12-23 only
    #    in scan 1 (12 votes each); both scans hold every pole's position, so both register with all 25 rows, and the
    #    lower rank wins the tie in inliers too.  Scan 1 (min_gap 1) votes 12 times for scan 0, onto its first row.
    s = seq([ident, mv(1, 0), mv(2, 1)], [R(12) + [p + NODESC for p in R(12, 25)],
                                          [p + NODESC for p in R(12)] + R(12, 24) + [24 + NODESC], R(24) + [24 + NODESC]])
    cases.append({"scans": s, "min_gap": 1, "candidates": 4, "want": {
        s + 1: {"loop": -1, "cand_scan": [s, -1, -1, -1], "cand_votes": [12, 0, 0, 0], "cand_status": [0, -1, -1, -1]},
        s + 2: {"loop": 0, "loop_scan": s, "n_inliers": 25, "cand_scan": [s, s + 1, -1, -1], "cand_votes": [12, 12, 0, 0],
                "cand_inliers": [25, 25, 0, 0], "cand_status": [2, 2, -1, -1]}}})
    # 2: the same pole in several earlier scans: scans 0, 1 and 2 each hold poles 0-16; the lowest row wins, so scan 0
    #    gets every vote of scan 4 (min_gap 2), and scans 1 and 2 none.
    s = seq([ident, mv(1, 0), mv(2, 0), mv(3, 0), mv(5, 0)], [R(17)] * 3 + [R(17, 25), R(17)])
    cases.append({"scans": s, "min_gap": 2, "candidates": 3, "want": {
        s + 4: {"loop": 0, "loop_scan": s, "n_inliers": 17, "cand_scan": [s, -1, -1], "cand_votes": [17, 0, 0],
                "cand_status": [2, -1, -1]}}})
    # 3: the top-voted candidate fails verification: scan 0 holds the descriptors of poles 0-19 but at moved positions
    #    (20 votes, no hypothesis survives); scan 1 holds every position of poles 0-22, with descriptors for 20-22 only
    #    (3 votes), and registers scan 3 with all 23 rows at rank 2.
    s = seq([ident, mv(1, 0), mv(2, 0), mv(3, 0)],
            [[p + MOVED for p in R(20)], [p + NODESC for p in R(20)] + R(20, 23), R(23, 25), R(23)])
    cases.append({"scans": s, "min_gap": 2, "candidates": 2, "want": {
        s + 3: {"loop": 1, "loop_scan": s + 1, "n_inliers": 23, "cand_scan": [s, s + 1], "cand_votes": [20, 3],
                "cand_status": [0, 2], "cand_inliers": [0, 23]}}})
    # 4: poles 21-24 also appear in sequence 0 with the same descriptors: they get no vote across sequences.  Fewer
    #    voted scans than candidates, rows without a descriptor (no vote), an empty scan, scans before min_gap.
    s = seq([ident, mv(1, 0), mv(2, 0), mv(3, 0)], [R(21, 25), [], [-1, 21], [21, 22, -1]])
    cases.append({"scans": s, "min_gap": 2, "candidates": 4, "want": {
        s: {"loop": -1, "cand_scan": [-1] * 4, "cand_status": [-1] * 4},
        s + 1: {"loop": -1, "cand_scan": [-1] * 4, "cand_status": [-1] * 4},
        s + 2: {"loop": -1, "cand_scan": [s, -1, -1, -1], "cand_votes": [1, 0, 0, 0], "cand_status": [0, -1, -1, -1]},
        s + 3: {"loop": -1, "cand_scan": [s, -1, -1, -1], "cand_votes": [2, 0, 0, 0], "cand_status": [1, -1, -1, -1]}}})
    # 5: an empty sequence, then a sequence of empty scans
    seq([], [])
    s = seq([ident, ident, ident], [[], [], []])
    cases.append({"scans": s, "min_gap": 1, "candidates": 1, "want": {
        s + 1: {"loop": -1, "cand_scan": [-1], "cand_status": [-1]}, s + 2: {"loop": -1, "cand_scan": [-1]}}})
    return (np.concatenate(rows), pole_rows(desc), np.array(ko, np.int64), np.array(so, np.int64), cases,
            np.array(pole, np.int64))


# ---- out-and-back paths ---------------------------------------------------------------------------------------------

def out_and_back(rng, n_out=15, n_back=15):
    """(n_out + n_back, 3) sensor poses (x, y, yaw): n_out scans forward at 0.5-1.5 m a step (up to 0.1 m sideways),
    then n_back scans back by 0.5-1.5 m a step, the first of them also moved sideways by up to 1.5 m; yaw jitters by up
    to 0.05 rad a step throughout, so the sensor keeps facing +x (the config 4 scene lies ahead of the origin)."""
    n = n_out + n_back
    poses = np.zeros((n, 3))
    for s in range(1, n):
        x, y, yaw = poses[s - 1]
        f, side, dyaw = rng.uniform(0.5, 1.5), rng.uniform(-0.1, 0.1), rng.uniform(-0.05, 0.05)
        if s >= n_out:
            f = -f
        if s == n_out:
            side = rng.uniform(-1.5, 1.5)
        poses[s] = (x + np.cos(yaw) * f - np.sin(yaw) * side, y + np.sin(yaw) * f + np.cos(yaw) * side, yaw + dyaw)
    return poses


def loop_sequence(synth, cfg, seq):
    """Out-and-back sequence `seq` of config `cfg`: seed (cfg, seq, 15) through the scene of scan 2000 + seq.
    -> points, scan_offsets, roll_pitch, poses"""
    poses = out_and_back(np.random.default_rng([cfg, seq, 15]))
    pts, offs, rp = synth.generate_poses(cfg, 2000 + seq, poses)
    return pts, offs, rp, poses


def between(poses, j, t):
    """Ground truth T(j)^-1 T(t) as {c, s, tx, ty}: scan t's levelled xy -> scan j's."""
    dyaw = poses[t, 2] - poses[j, 2]
    dx, dy = poses[t, 0] - poses[j, 0], poses[t, 1] - poses[j, 1]
    c0, s0 = np.cos(poses[j, 2]), np.sin(poses[j, 2])
    return np.array([np.cos(dyaw), np.sin(dyaw), c0 * dx + s0 * dy, -s0 * dx + c0 * dy])


def revisits(poses, min_gap):
    """Scans t with an earlier scan j <= t - min_gap within 2 m and 10 deg in the ground truth."""
    out = []
    for t in range(len(poses)):
        for j in range(t - min_gap + 1):
            if np.hypot(*(poses[t, :2] - poses[j, :2])) <= 2.0 and abs(poses[t, 2] - poses[j, 2]) <= np.radians(10.0):
                out.append(t)
                break
    return out


@functools.lru_cache(maxsize=None)
def oracle_chain(cfg, kind, seq):
    """Oracle pipeline on sequence `seq` of config `cfg`, `kind` "loop" (out-and-back) or "forward"
    (register_cases.sequence) -> ko, kp, descriptors, poses."""
    from feature_extraction_b200 import synth
    from oracle import oracle_binding as ob
    pts, offs, rp, poses = (loop_sequence if kind == "loop" else sequence)(synth, cfg, seq)
    ko, kpts, d, _ = ob.process_batch(oracle_params(ob, cfg), pts, offs, rp, mode=0, n_threads=8)
    return ko, kpts, d, poses


def inverse(a):
    return np.array([a[0], -a[1], -(a[0] * a[2] + a[1] * a[3]), a[1] * a[2] - a[0] * a[3]])


def choose(o, K):
    """The loop of every scan when only the first K ranks of `o` (a call with more candidates) are kept: the choice
    rule applied to them.  Ranks do not depend on `candidates`, and a candidate's verification depends only on its
    pair of scans, so this is what a call with K candidates returns."""
    loop = np.full(len(o["loop"]), -1)
    for t in range(len(loop)):
        best = -1
        for k in range(K):
            if o["cand_status"][t, k] == 2 and (best < 0 or o["cand_inliers"][t, k] > o["cand_inliers"][t, best]):
                best = k
        loop[t] = best
    return loop


@functools.lru_cache(maxsize=None)
def oracle_loops(cfg, kind, seq, min_gap, candidates, threads=8):
    """feo_loop_closures and feo_odometry (W = 2) on oracle_chain(cfg, kind, seq) -> loops, odometry."""
    from match_oracle import binding as mo
    ko, kpts, d, _ = oracle_chain(cfg, kind, seq)
    o = mo.loop_closures(kpts, d, ko, [0, len(ko) - 1], min_gap, candidates, n_threads=threads)
    best = mo.match_descriptors(d, d, ko[1:], ko[:-1], n_threads=threads)[0] if len(ko) > 2 else np.zeros(0, np.int64)
    return o, mo.odometry(kpts, ko, best, [0, len(ko) - 1], 2)


def evaluate(cfg, min_gap, candidates, n_seq=20, threads=8, from_candidates=None):
    """The oracle loop closures on n_seq out-and-back and n_seq forward sequences.  -> dict of revisits, found (revisit
    scans with a loop), wrong (loops anywhere more than 0.5 m or 2 deg off T(j)^-1 T(t)), and per found loop its
    translation (m) and yaw (deg) error beside those of odometry's own pose_j^-1 pose_t (W = 2) for the same pair.
    from_candidates: take the loops from calls with that many candidates (choose())."""
    from odometry_cases import compose
    r = {"revisits": 0, "found": 0, "wrong": 0, "dt": [], "dy": [], "odo_dt": [], "odo_dy": []}
    for kind in ("loop", "forward"):
        for i in range(n_seq):
            poses = oracle_chain(cfg, kind, i)[3]
            o, odo = oracle_loops(cfg, kind, i, min_gap, from_candidates or candidates, threads)
            loop = choose(o, candidates) if from_candidates else o["loop"]
            rev = set(revisits(poses, min_gap)) if kind == "loop" else set()
            r["revisits"] += len(rev)
            for t in np.nonzero(loop >= 0)[0]:
                j = int(o["cand_scan"][t, loop[t]])
                truth = between(poses, j, t)
                dt, dy = errors(o["cand_pose"][t, loop[t]], truth)
                odt, ody = errors(compose(inverse(odo["pose"][j]), odo["pose"][t]), truth)
                if dt[0] > 0.5 or np.degrees(dy[0]) > 2.0:
                    r["wrong"] += 1
                r["found"] += int(t in rev)
                r["dt"].append(dt[0])
                r["dy"].append(np.degrees(dy[0]))
                r["odo_dt"].append(odt[0])
                r["odo_dy"].append(np.degrees(ody[0]))
    r["fraction"] = r["found"] / r["revisits"] if r["revisits"] else 0.0
    return r
