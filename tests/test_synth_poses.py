"""synth.generate_poses: one scene rendered from several sensor poses."""
import numpy as np
import pytest

from register_cases import apply, oracle_params, relative, sequence


@pytest.mark.parametrize("cfg", [1, 2, 3, 4, 5])
def test_scan_0_at_the_identity_is_generate(synth, cfg):
    a = synth.generate(cfg, 1, scan_index_base=7)
    b = synth.generate_poses(cfg, 7, [[0.0, 0.0, 0.0], [1.0, 0.2, 0.05]])
    n0 = int(a[1][1])
    assert np.array_equal(a[0].view(np.uint32), b[0][:n0].view(np.uint32))
    assert b[1][1] == n0
    assert np.array_equal(a[2][0], b[2][0])
    if cfg != 1:  # config 1 has a fixed roll and pitch
        assert not np.array_equal(b[2][0], b[2][1])  # scan 1 draws them from a stream of its own


def test_keypoints_of_consecutive_scans_coincide_under_the_ground_truth(ob, synth):
    """The oracle's keypoints of scan s, moved into scan s-1 by the ground-truth motion, lie within 0.5 m of a keypoint
    of scan s-1 for most keypoints (poles leave the crop box and the field of view as the sensor moves)."""
    near = total = 0
    for seq in range(2):
        pts, offs, rp, poses = sequence(synth, 4, seq)
        ko, kp, _, _ = ob.process_batch(oracle_params(ob, 4), pts, offs, rp, mode=0, n_threads=8)
        truth = relative(poses)
        for s in range(1, len(ko) - 1):
            w = apply(truth[s - 1], kp[ko[s]:ko[s + 1], :2])
            ref = kp[ko[s - 1]:ko[s], :2].astype(np.float64)
            if len(w) == 0 or len(ref) == 0:
                continue
            d = np.sqrt(((w[:, None] - ref[None]) ** 2).sum(-1)).min(axis=1)
            near += int((d < 0.5).sum())
            total += len(w)
    print("config 4: %d of %d keypoints (%.3f) within 0.5 m of a keypoint of the previous scan" % (near, total, near / total))
    assert total > 500 and near / total > 0.75
