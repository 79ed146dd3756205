"""Constructed scans for the boundary kinds 4-9 of fe_enable_boundary_report_all (include/fe_b200.h), shared by
the CPU oracle test and its GPU twin.  roll = pitch = 0, so the levelled cloud is the input.

case(ob, kind, offset) -> (params, points, scan_offsets, roll_pitch): one scan whose decision of `kind` lies
`offset` metres from its boundary (about 4e-7 m: counted at eps 1e-6; 1e-3 m: not counted).
"""
import numpy as np

DEG = 0.017453292519943295
EPS = 1e-6
NEAR = 4e-7      # distance of the constructed decision from its boundary
FAR = 1e-3
RANGE = 10.0     # of the ring-window point and the cluster


def params(ob, desc=False):
    P = ob.node_default()  # cluster_tolerance 0.65, sizes 5..50, radius threshold 0.15, one detection channel
    P.z_max = 1.0
    P.estimate_descriptors = 1 if desc else 0
    return P


def _scan(pts):
    pts = np.asarray(pts, np.float32).reshape(-1, 4)
    return pts, np.array([0, len(pts)], np.int64), np.zeros((1, 2), np.float64)


def crop_point(z_over, x=5.0):
    """[4] one point z_over metres above the crop box's z_max of 1.0 (negative: inside)."""
    return [x, 0.0, float(np.float32(1.0 + z_over)), 0.0]


def ring_point(d_deg):
    """[5] one point RANGE metres out whose elevation is 2 deg + d_deg: the end of ring windows [0, 2] and [2, 4]."""
    el = np.radians(2.0 + d_deg)
    return [RANGE * np.cos(el), 0.0, RANGE * np.sin(el), 0.0]


def cluster(span):
    """[6] six points of the -1 deg ring along y whose xy diameter is `span` (the gate is 2 x 0.15 = 0.3 m)."""
    y = np.linspace(-0.15, -0.15 + span, 6)
    y[-1] = -0.15 + span
    z = -RANGE * np.tan(np.radians(1.0))
    return [[RANGE, float(v), z, 0.0] for v in y]


def keypoint_of_cluster(ob, P):
    """the keypoint the gated cluster of diameter 0.29 m becomes (the origin of the 3DSC cases)"""
    pts, offs, rp = _scan(cluster(0.29))
    ko, kp, _, _ = ob.process_batch(P, pts, offs, rp, mode=0, want_desc=False)
    assert len(kp) == 1
    return kp[0]


def neighbour(ob, kind, offset):
    """[7-9] a surface point added to the 0.29 m cluster, placed relative to its keypoint o:
    7: straight above at radii[10] + offset; 8: at 1.45 m with theta = theta_div[1] + offset / 1.45 m (in x-z);
    9: straight above at 0.9 m, moved `offset` in x (rho = 0 when offset == 0)."""
    P = params(ob, desc=True)
    o = keypoint_of_cluster(ob, P).astype(np.float64)
    radii, theta, _, _ = ob.sc3d_tables(P.descriptor_radius)
    if kind == 7:
        q = [o[0], o[1], o[2] + float(radii[10]) + offset]
    elif kind == 8:
        # x (float spacing 1e-6 m out here) is the same for every offset; the angle moves through z (1e-7 m)
        r = 1.45
        th0 = np.radians(float(theta[1]))
        qx = np.float32(o[0] + r * np.sin(th0))
        dx = float(qx - np.float32(o[0]))
        q = [float(qx), o[1], o[2] + dx / np.tan(th0 + offset / r)]
    else:
        q = [o[0] + offset, o[1], o[2] + 0.9]
    return P, q + [0.0]


def case(ob, kind, offset):
    if kind == 4:
        return (params(ob),) + _scan([crop_point(offset)])
    if kind == 5:
        return (params(ob),) + _scan([ring_point(offset / (RANGE * DEG))])
    if kind == 6:
        return (params(ob),) + _scan(cluster(0.3 + offset))
    P, q = neighbour(ob, kind, offset)
    return (P,) + _scan(cluster(0.29) + [q])


def base_case(ob, kind):
    """the scan of `case` without the constructed decision (kinds 7-9: the cluster alone)"""
    if kind in (7, 8, 9):
        return (params(ob, desc=True),) + _scan(cluster(0.29))
    return (params(ob),) + _scan(np.zeros((0, 4)))
