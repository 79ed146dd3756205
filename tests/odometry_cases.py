"""Inputs of the odometry tests (include/fe_b200.h, "odometry"): constructed sequences whose links are known exactly,
the contract's motion algebra in numpy, and the oracle chain on the synthetic sequences of register_cases, cached
per sequence so that several windows reuse one pipeline and match."""
import functools

import numpy as np

from register_cases import C24, S7, errors, kp, oracle_params, relative, sequence

IDENTITY = np.array([1.0, 0.0, 0.0, 0.0])


def compose(a, b):
    """The contract's compose(A, B), operation by operation."""
    return np.array([a[0] * b[0] - a[1] * b[1], a[1] * b[0] + a[0] * b[1], (a[0] * b[2] - a[1] * b[3]) + a[2],
                     (a[1] * b[2] + a[0] * b[3]) + a[3]])


def chain(motion, source):
    """pose_t = compose(pose_{t-1}, motion_t) within each sequence (a scan with source 0 starts one)."""
    pose = np.zeros_like(motion)
    for s in range(len(motion)):
        pose[s] = IDENTITY if source[s] == 0 else compose(pose[s - 1], motion[s])
    return pose


# Poles of the constructed scenes: 25 points at multiples of 25 m, so that frames turned by (24/25, 7/25) and moved
# by multiples of 25 m (or not turned and moved by whole metres) see every pole at integer coordinates.
POLES = 25.0 * np.array([[a, b] for a, b in
                         [(-4, -3), (-3, 1), (-2, 4), (-1, -2), (0, 3), (1, -4), (2, 2), (3, -1), (4, 1), (-4, 2),
                          (-3, -4), (-2, -1), (-1, 1), (0, -3), (1, 4), (2, -2), (3, 3), (4, -4), (-4, 4), (-3, -2),
                          (-1, 4), (0, 0), (1, 1), (2, -4), (4, 3)]], np.float64)


def _in_frame(frame, xy):
    """Scene xy -> the frame's xy, for a frame (c, s, tx, ty) that maps its xy into the scene."""
    c, s, tx, ty = frame
    dx, dy = xy[:, 0] - tx, xy[:, 1] - ty
    return np.stack([c * dx + s * dy, -s * dx + c * dy], axis=1)


def constructed():
    """Sequences with known links under the default registration parameters (min_inliers = 16).
    -> kp, keypoint_offsets, best, sequence_offsets, and per sequence a dict of what the contract implies: `scans`
    (absolute scan of local scan 0) and `want(W)` -> {absolute scan: {field: value}}.  Rows carry their pole's index in
    `pole` (absolute row -> pole)."""
    rows, ko, so, seqs, pole, best = [], [0], [0], [], [], []
    R = lambda *a: list(range(*a))  # noqa: E731

    def seq(frames, visible, want, first_best=None):
        s0 = len(ko) - 1
        for t, (frame, vis) in enumerate(zip(frames, visible)):
            xy = _in_frame(frame, POLES[vis]) if len(vis) else np.zeros((0, 2))
            rows.append(kp(xy))
            start = ko[-1]
            ko.append(start + len(vis))
            if s0 + t == 0:
                pass  # the batch's first scan has no `best` entries
            elif t == 0:
                best.extend(first_best(start, len(vis)) if first_best else [-1] * len(vis))
            else:
                prev = {p: ko[-3] + i for i, p in enumerate(visible[t - 1])}
                best.extend(prev.get(p, -1) for p in vis)
            pole.extend(vis)
        so.append(len(ko) - 1)
        seqs.append({"scans": s0, "want": want})

    rot = lambda tx, ty: np.array([C24, S7, tx, ty])  # noqa: E731
    mv = lambda tx, ty: np.array([1.0, 0.0, tx, ty])  # noqa: E731

    # 0: a pole (16) seen in scans 0 and 2 but not 1: W = 1 leaves link 2 at 15 inliers, W >= 2 registers it with 16
    seq([IDENTITY, rot(25, 0), rot(50, 25)], [R(17), R(16), R(15) + [16]],
        lambda W: {1: {"source": 1, "n_inliers": 16},
                   2: {"source": 1, "n_inliers": 16} if W >= 2 else {"source": 2, "status": 1, "n_inliers": 15}})
    # 1: link 2 is predicted (15 inliers) and equals motion 1 (constant velocity, here also the truth); link 3 then sees
    #    pole 16, which only scans 0 and 1 hold: the predicted link cuts the window, so link 3 scores 16 at every W,
    #    not 17.  Its first scan's `best` points into sequence 0, as the matcher leaves it.
    seq([IDENTITY, mv(3, -2), mv(6, -4), rot(25, 25)], [R(17), R(17), R(15) + [20], R(15) + [20, 16]],
        lambda W: {1: {"source": 1, "n_inliers": 17}, 2: {"source": 2, "status": 1, "n_inliers": 15},
                   3: {"source": 1, "n_inliers": 16}},
        first_best=lambda start, n: [start - 1 - (i % 3) for i in range(n)])
    # 2: link 1 has 3 inliers: predicted, the identity at t = 1.  First-scan `best` entries that no scan holds.
    seq([IDENTITY, mv(2, 1)], [R(17), R(3)],
        lambda W: {1: {"source": 2, "status": 1, "n_inliers": 3}},
        first_best=lambda start, n: [12345678, -7] + [-1] * (n - 2))
    # 3: an empty sequence; 4: a sequence of one scan
    seq([], [], lambda W: {})
    seq([IDENTITY], [R(6)], lambda W: {})
    # 5: empty scans: nothing to register against (link 1), nothing to register (link 2), then an empty window again
    seq([IDENTITY, mv(1, 0), mv(2, 0), mv(3, 0)], [[], R(17), [], R(17)],
        lambda W: {1: {"source": 2, "status": 0}, 2: {"source": 2, "status": 0}, 3: {"source": 2, "status": 0}})
    return (np.concatenate(rows), np.array(ko, np.int64), np.array(best, np.int64), np.array(so, np.int64), seqs,
            np.array(pole, np.int64))


def scan_pairs_best(ko, best, so):
    """`best` with the entries of first scans set to -1, as fe_register_matches on scan s against s - 1 accepts it."""
    b = best.copy()
    for f in so[1:-1]:
        if f < len(ko) - 1:
            b[ko[f] - ko[1]:ko[f + 1] - ko[1]] = -1
    return b


# ---- the synthetic sequences ----------------------------------------------------------------------------------------

def to_first(poses):
    """Ground truth T(0)^-1 T(s) for every scan s as (n, 4) {c, s, tx, ty}: scan s's levelled xy -> scan 0's."""
    dyaw = poses[:, 2] - poses[0, 2]
    dx, dy = poses[:, 0] - poses[0, 0], poses[:, 1] - poses[0, 1]
    c0, s0 = np.cos(poses[0, 2]), np.sin(poses[0, 2])
    return np.stack([np.cos(dyaw), np.sin(dyaw), c0 * dx + s0 * dy, -s0 * dx + c0 * dy], axis=1)


@functools.lru_cache(maxsize=None)
def oracle_chain(cfg, seq):
    """Oracle pipeline and matcher on sequence `seq` of config `cfg` -> ko, kp, best (scan s against s - 1), poses."""
    from feature_extraction_b200 import synth
    from match_oracle import binding as mo
    from oracle import oracle_binding as ob
    pts, offs, rp, poses = sequence(synth, cfg, seq)
    ko, kpts, d, _ = ob.process_batch(oracle_params(ob, cfg), pts, offs, rp, mode=0, n_threads=8)
    best = mo.match_descriptors(d, d, ko[1:], ko[:-1], n_threads=8)[0]
    return ko, kpts, best, poses


def evaluate(cfg, window, n_seq=20):
    """The oracle odometry on n_seq sequences of 20 scans.  -> registered fraction of links, wrong links (registered,
    more than 0.5 m or 2 deg off the truth), end-point translation (m) and yaw (deg) errors per sequence."""
    from match_oracle import binding as mo
    reg, wrong, dt_end, dy_end = [], 0, [], []
    for i in range(n_seq):
        ko, kpts, best, poses = oracle_chain(cfg, i)
        o = mo.odometry(kpts, ko, best, [0, len(ko) - 1], window)
        ok = o["source"][1:] == 1
        dt, dy = errors(o["motion"][1:], relative(poses))
        wrong += int(((dt[ok] > 0.5) | (np.degrees(dy[ok]) > 2.0)).sum())
        reg.append(ok)
        et, ey = errors(o["pose"][-1], to_first(poses)[-1])
        dt_end.append(et[0])
        dy_end.append(np.degrees(ey[0]))
    return float(np.concatenate(reg).mean()), wrong, np.array(dt_end), np.array(dy_end)
