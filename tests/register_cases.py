"""Inputs of the registration tests (include/fe_b200.h, "registration"): sensor paths through one synthetic scene with
their ground-truth relative motions, and constructed groups whose answer is known exactly."""
import numpy as np

# (c, s) = (24/25, 7/25): a yaw of 16.26 deg that maps points with coordinates in multiples of 25 m onto integers, so
# that the float keypoints of both sides are exact and the planted motion is recovered to the last bits.
C24, S7 = 24.0 / 25.0, 7.0 / 25.0


def path(rng, n_scans=20):
    """(n_scans, 3) sensor poses (x, y, yaw) in the scene frame: from the origin, each step 0.5-1.5 m forward, up to
    0.1 m sideways and up to 0.05 rad of yaw."""
    poses = np.zeros((n_scans, 3))
    for s in range(1, n_scans):
        x, y, yaw = poses[s - 1]
        f, side, dyaw = rng.uniform(0.5, 1.5), rng.uniform(-0.1, 0.1), rng.uniform(-0.05, 0.05)
        poses[s] = (x + np.cos(yaw) * f - np.sin(yaw) * side, y + np.sin(yaw) * f + np.cos(yaw) * side, yaw + dyaw)
    return poses


def relative(poses):
    """Ground truth T(s-1)^-1 T(s) for s = 1..n-1 as (n-1, 4) {c, s, tx, ty}: scan s's levelled xy -> scan s-1's."""
    p0, p1 = poses[:-1], poses[1:]
    dyaw = p1[:, 2] - p0[:, 2]
    dx, dy = p1[:, 0] - p0[:, 0], p1[:, 1] - p0[:, 1]
    c0, s0 = np.cos(p0[:, 2]), np.sin(p0[:, 2])
    return np.stack([np.cos(dyaw), np.sin(dyaw), c0 * dx + s0 * dy, -s0 * dx + c0 * dy], axis=1)


def apply(pose, xy):
    c, s, tx, ty = pose
    xy = np.asarray(xy, np.float64)
    return np.stack([c * xy[..., 0] - s * xy[..., 1] + tx, s * xy[..., 0] + c * xy[..., 1] + ty], axis=-1)


def errors(pose, truth):
    """-> translation error (m) and yaw error (rad) of estimated motions against the ground truth, per row."""
    pose, truth = np.atleast_2d(pose), np.atleast_2d(truth)
    dt = np.hypot(pose[:, 2] - truth[:, 2], pose[:, 3] - truth[:, 3])
    dyaw = np.abs(np.arctan2(pose[:, 1] * truth[:, 0] - pose[:, 0] * truth[:, 1],
                             pose[:, 0] * truth[:, 0] + pose[:, 1] * truth[:, 1]))
    return dt, dyaw


def oracle_params(ob, cfg):
    P = ob.launch_playback() if cfg == 1 else ob.node_default()
    if cfg == 4:
        P.descriptor_radius = 5.0
    return P


def sequence(synth, cfg, seq, n_scans=20):
    """Sequence `seq` of config `cfg`: a path from seed (cfg, seq) through the scene of scan 1000 + seq.
    -> points, scan_offsets, roll_pitch, poses"""
    poses = path(np.random.default_rng([cfg, seq]), n_scans)
    pts, offs, rp = synth.generate_poses(cfg, 1000 + seq, poses)
    return pts, offs, rp, poses


def kp(xy):
    """(n, 2) positions -> (n, 4) float32 keypoints (z = -1, elevation 0)."""
    xy = np.asarray(xy, np.float64).reshape(-1, 2)
    return np.concatenate([xy, np.full((len(xy), 1), -1.0), np.zeros((len(xy), 1))], axis=1).astype(np.float32)


PARAMS = dict(inlier_radius=0.5, min_separation=1.0, max_hypotheses=512, min_inliers=3, refine_iterations=4)


def constructed():
    """Groups with a known answer.  -> query keypoints, reference keypoints, best, query_offsets, ref_offsets, and per
    group a dict of what the contract implies with PARAMS.
    Query rows start at row 2 (rows 0-1 belong to no group); reference rows at row 1."""
    Q, R, B, qo, ro, want = [np.zeros((2, 2))], [np.zeros((1, 2))], [], [2], [1], []

    def group(q_xy, r_xy, best_local, **w):
        r0 = ro[-1]
        Q.append(np.asarray(q_xy, np.float64).reshape(-1, 2))
        R.append(np.asarray(r_xy, np.float64).reshape(-1, 2))
        B.extend(-1 if b < 0 else r0 + b for b in best_local)
        qo.append(qo[-1] + len(Q[-1]))
        ro.append(ro[-1] + len(R[-1]))
        want.append(w)

    grid = 25.0 * np.array([[a, b] for a in range(-2, 3) for b in range(-1, 2)], np.float64)  # 15 points
    planted = np.array([C24, S7, 3.0, -2.0])
    ref = apply(planted, grid)
    # 0: planted motion, 10 correct matches, 3 wrong ones, 2 query rows without a descriptor (best -1) but on a
    #    reference row, 2 query rows far from everything
    best = list(range(10)) + [12, 10, 11] + [-1, -1, -1, -1]
    qxy = np.concatenate([grid, [[500.0, 500.0], [-500.0, 40.0]]])
    group(qxy, ref, best, pose=planted, status=2, n_inliers=15, assoc_of=list(range(15)) + [-1, -1])
    # 1: a single correspondence (n_c = 1): no hypothesis
    group(grid[:3], ref[:3], [0, -1, -1], status=0, n_hypotheses=0)
    # 2: every pair closer than min_separation: all rejected
    near = np.array([[10.0, 10.0], [10.3, 10.1], [10.1, 10.4], [10.2, 10.2]])
    group(near, near + 5.0, [0, 1, 2, 3], status=0, n_hypotheses=0)
    # 3: two matches onto one reference row: that pair has lv = 0 and is rejected; so are the two other pairs of the
    #    wrongly matched row 3, whose lengths change by 25 m and 10 m; 3 of 6 pairs survive, and geometry puts row 3 on
    #    its true reference row
    group(grid[:4], ref[:4], [0, 1, 2, 2], status=2, n_hypotheses=3, n_inliers=4, pose=planted)
    # 4: P = 40*39/2 = 780 > 512 hypotheses: 512 are tried, every one of them valid
    g40 = np.array([[5.0 * a, 7.0 * b] for a in range(8) for b in range(5)])
    group(g40, g40 + [1.0, 2.0], list(range(40)), status=2, n_hypotheses=512, n_inliers=40,
          pose=np.array([1.0, 0.0, 1.0, 2.0]))
    # 5: a tie: rows 0-2 fit motion M1 (shift +1 m in x), rows 3-5 motion M2 (shift +30 m in y); every pair across
    #    the two sets changes length by far more than 1 m and is rejected; both motions score 3, and the lower h (a pair
    #    of rows 0-2) wins
    a = np.array([[0.0, 0.0], [10.0, 0.0], [0.0, 10.0]])
    b = np.array([[40.0, 40.0], [50.0, 40.0], [40.0, 50.0]])
    group(np.concatenate([a, b]), np.concatenate([a + [1.0, 0.0], b + [0.0, 30.0]]), [0, 1, 2, 3, 4, 5], status=2,
          n_inliers=3, n_hypotheses=6, pose=np.array([1.0, 0.0, 1.0, 0.0]), assoc_of=[0, 1, 2, -1, -1, -1])
    # 6: the tie the other way round: M2's rows first
    group(np.concatenate([b, a]), np.concatenate([b + [0.0, 30.0], a + [1.0, 0.0]]), [0, 1, 2, 3, 4, 5], status=2,
          n_inliers=3, n_hypotheses=6, pose=np.array([1.0, 0.0, 0.0, 30.0]), assoc_of=[0, 1, 2, -1, -1, -1])
    # 7: empty group (no query and no reference rows)
    group(np.zeros((0, 2)), np.zeros((0, 2)), [], status=0, n_hypotheses=0)
    # 8: queries but no reference rows
    group(grid[:3], np.zeros((0, 2)), [-1, -1, -1], status=0, n_hypotheses=0)
    # 9: NaN-descriptor rows (best = -1) only, apart from two matches: the two fix the motion, all five are inliers
    group(grid[:5], ref[:5], [0, -1, -1, 3, -1], status=2, n_hypotheses=1, n_inliers=5, pose=planted,
          assoc_of=[0, 1, 2, 3, 4])
    # 10: two matches whose lengths differ by 1 m >= 2 * radius: rejected
    group([[0.0, 0.0], [10.0, 0.0]], [[0.0, 0.0], [11.0, 0.0]], [0, 1], status=0, n_hypotheses=0)
    q = kp(np.concatenate(Q))
    r = kp(np.concatenate(R))
    return q, r, np.array(B, np.int64), np.array(qo, np.int64), np.array(ro, np.int64), want


def hypothesis_pairs(n_c, max_hypotheses):
    """The contract's hypothesis map: pair index floor(h*P/H) for h in [0, H)."""
    P = n_c * (n_c - 1) // 2
    H = min(P, max_hypotheses)
    return [h * P // H for h in range(H)]
