"""The device's 3DSC descriptors against the independent reference of sc3d_cases.py and bit for bit against the CPU
oracle, at every K4d tier (block per keypoint, warp per keypoint, the three k_desc_hist instantiations, bin groups and
the order-free bin), at K4b's per-warp neighbour list (one warp listing exactly MARK_WCAP = 512 and 513 entries), with
d2 ties whose summation order is visible, and at both per-scan limits (65,536 keypoints with neighbours, 2^20
points)."""
import numpy as np
import pytest

import sc3d_cases as sc
from util import bits_equal, to_fe_params

pytestmark = pytest.mark.gpu
F32 = np.float32
R = 2.5

# exact neighbour counts at every K4d tier boundary: DW_CAP 256, DCAP 1536, DCAP_M 4096, DCAP_L 8192 (511-513 spread
# over the sphere's grid rows leave every K4b warp far below its list capacity; test_one_warp_at_its_list_capacity
# puts a single warp there)
LADDER = [255, 256, 257, 511, 512, 513, 1535, 1536, 1537, 4095, 4096, 4097, 8191, 8192, 8193, 20000]


def _node(ob, **kw):
    from feature_extraction_b200 import FeatureExtractionNode
    lim = dict(max_points=1 << 21, max_scans=64, max_keypoints=1 << 12)
    lim.update(kw)
    return FeatureExtractionNode(to_fe_params(ob.node_default()), **lim)


def _check(cloud, kps, got, axis_offset=0):
    return sc.check_descriptors_against_reference(cloud, kps, R, got, axis_offset)


# ---------------------------------------------------------------------------------------------------------------
# estimateDescriptors
# ---------------------------------------------------------------------------------------------------------------
def test_tier_ladder_through_estimate_descriptors(ob):
    rng = np.random.default_rng(11)
    counts = [0, 1] + LADDER
    kps, parts = [], []
    for i, n in enumerate(counts):
        c = (F32(8.0 * (i % 6)), F32(8.0 * (i // 6)), F32(0.25))
        kps.append([c[0], c[1], c[2], 0])
        parts.append(sc.with_count(rng, c, R, n))
    cloud = np.concatenate(parts)
    kps = np.array(kps, F32)
    d_o, _, nn = ob.estimate_descriptors(ob.node_default(), cloud, kps, mode=1)
    assert list(nn) == counts
    nd = _node(ob)
    d = nd.estimateDescriptors(cloud, kps)
    assert bits_equal(d, d_o)
    st = _check(cloud, kps, d)
    assert st["rows"] == len(counts) - 1 and st["ambiguous"] <= 1e-3 * st["contributions"], st
    assert nd.batchStats()["descriptors_unordered"] == 0
    print("\nestimateDescriptors ladder: ambiguous share %.1e of %d contributions" % (st["ambiguous"] / st["contributions"],
                                                                               st["contributions"]))
    nd.close()


def test_65536_keypoints_with_neighbours_per_scan_and_one_more_is_refused(ob):
    from feature_extraction_b200 import FeatureExtractionError, _native
    n = 1 << 16
    g = np.arange(n + 1)
    grid = np.stack([(g % 256) * 3.0, (g // 256) * 3.0, np.zeros(n + 1), np.zeros(n + 1)], axis=1).astype(F32)
    # the last four keypoints get real neighbourhoods: their axes are the last entries of the table
    rng = np.random.default_rng(61)
    cloud = np.concatenate([grid[:n + 1]] + [sc.with_count(rng, grid[i, :3], R, 300) for i in range(n - 4, n)])
    kps = grid[:n]
    nd = _node(ob, max_keypoints=1 << 17)
    d = nd.estimateDescriptors(cloud, kps)
    d_o, _, nn = ob.estimate_descriptors(ob.node_default(), cloud, kps, mode=1)
    assert (nn >= 1).all() and (nn[n - 4:] > 300).all() and bits_equal(d, d_o)
    assert (d[:n - 300] == 0).all()
    st = _check(cloud, kps[n - 8:], d[n - 8:], axis_offset=n - 8)   # every earlier keypoint drew an axis
    assert st["rows"] == 8 and st["contributions"] >= 1200
    # keypoints without a neighbour do not count: 65,536 described keypoints plus NaN and far-away ones are accepted
    extra = np.array([[np.nan, 0, 0, 0], [1e4, 1e4, 0, 0], [np.inf, 0, 0, 0]], F32)
    kx = np.concatenate([extra[:1], kps[:1000], extra[1:2], kps[1000:], extra[2:]])
    dx = nd.estimateDescriptors(cloud, kx)
    assert bits_equal(dx, ob.estimate_descriptors(ob.node_default(), cloud, kx, mode=1)[0])
    assert np.isnan(dx[[0, 1001, n + 2]]).all() and bits_equal(dx[n - 2:n + 2], d[n - 4:])
    with pytest.raises(FeatureExtractionError) as e:
        nd.estimateDescriptors(cloud, grid)                    # 65,537 keypoints with a neighbour
    assert e.value.status == _native.FE_ERR_CAPACITY
    # the context stays usable
    small = cloud[:300]
    assert bits_equal(nd.estimateDescriptors(small, small), ob.estimate_descriptors(ob.node_default(), small, small)[0])
    nd.close()


# ---------------------------------------------------------------------------------------------------------------
# processBatch: one pole per scan plus clutter outside the crop box within R of its keypoint
# ---------------------------------------------------------------------------------------------------------------
def pole(x0=1.0, y0=0.0):
    """Six points per ring on a 5 cm circle at range ~x0: one ring cluster per ring, merged into one keypoint."""
    pts = []
    for r in range(16):
        el = np.deg2rad(-15.0 + 2.0 * r)
        for a in range(6):
            t = 2 * np.pi * a / 6
            x, y = x0 + 0.05 * np.cos(t), y0 + 0.05 * np.sin(t)
            pts.append([x, y, np.hypot(x, y) * np.tan(el), 0.0])
    return np.array(pts, F32)


def clutter(rng, kp, n, lo=0.15, hi=0.97, box=None, groups=(), yslab=None):
    """n points within R of keypoint kp (exact predicate) behind the crop box (x <= -0.01): never clustered, but
    neighbours of the keypoint.  box: optional (r, theta, phi) ranges in (m, deg, deg about +x) to sample from; groups:
    azimuths (deg about +x) of tie groups (sc3d_cases.tie_group) whose outer shell, elevation band and a 35 deg wedge
    around them (more than the group's bin) stay empty; yslab: (y0, y1) to keep y in."""
    out, R2f = [np.zeros((0, 3), F32)], sc.radius_sq_float(R)
    while sum(len(o) for o in out) < n:
        m = 4 * n + 64
        if box is None:
            p = sc.ball_points(rng, kp[:3], m, lo * R, hi * R)
        else:
            (r0, r1), (t0, t1), (f0, f1) = box
            r = rng.uniform(r0, r1, m)
            t = np.deg2rad(rng.uniform(t0, t1, m))
            f = np.deg2rad(rng.uniform(f0, f1, m))
            p = (kp[:3].astype(np.float64) + np.stack([r * np.sin(t) * np.cos(f), r * np.sin(t) * np.sin(f),
                                                        r * np.cos(t)], 1)).astype(F32)
        keep = (p[:, 0] <= -0.01) & (sc.d2_f32(kp[:3], p) < R2f)
        if yslab is not None:
            keep &= (p[:, 1] >= yslab[0]) & (p[:, 1] <= yslab[1])
        v = p.astype(np.float64) - np.asarray(kp, np.float64)[:3]
        r = np.linalg.norm(v, axis=1)
        az = np.rad2deg(np.arctan2(v[:, 1], v[:, 0]))
        for g in groups:
            near = (r > 1.7) & (np.abs(v[:, 2]) < 0.3 * r) & (np.abs((az - g + 180.0) % 360.0 - 180.0) < 35.0)
            keep &= ~near
        out.append(p[keep])
    p = np.concatenate(out)[:n]
    return np.concatenate([p, np.zeros((n, 1), F32)], axis=1)


@pytest.fixture(scope="module")
def pole_kp(ob):
    P = ob.node_default()
    r = ob.process_scan(P, pole(), 0.0, 0.0, mode=1)
    assert len(r["keypoints"]) == 1
    return r["keypoints"][0], len(pole())


@pytest.fixture(scope="module")
def lut():
    from oracle import oracle_binding
    return oracle_binding.sc3d_tables(R)[3]


def ladder_scans(pole_kp, counts, seed):
    """One scan per count: the pole, clutter to make the keypoint's neighbour count exactly `count` and, at the end of
    the scan, a tie group (sc3d_cases.tie_group) behind the crop box.  -> points, offsets, roll_pitch, and per scan the
    scan-local indices (B, A) of the tie."""
    kp, npole = pole_kp
    rng = np.random.default_rng(seed)
    grp = sc.tie_group(kp, 180.0)
    assert all((grp[k][:, 0] < 0).all() for k in grp)
    scans, tie = [], []
    for n in counts:
        c = clutter(rng, kp, n - npole - 3, groups=(180.0,))
        s = np.concatenate([pole(), c, grp["extra"], grp["C"], grp["B"], grp["A"]])
        tie.append((len(s) - 2, len(s) - 1))
        scans.append(s)
    offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
    return np.concatenate(scans), offs, np.zeros((len(scans), 2)), tie


def _oracle_scans(ob, pts, offs):
    P = ob.node_default()
    return [ob.process_scan(P, pts[offs[s]:offs[s + 1]], 0.0, 0.0, mode=1) for s in range(len(offs) - 1)]


def _assert_tie_order(ref, lut, got_row, b_idx, a_idx):
    """The tie (B, A) lands in one unambiguous bin whose float sum changes if the two swap places, and the device's bin
    is the sum in (d2, index) order."""
    det = ref["detail"][0]
    t = {int(i): k for k, i in enumerate(det["idx"])}
    ta, tb = t[a_idx], t[b_idx]
    assert det["d2"][ta] == det["d2"][tb] and det["rho"][ta] != det["rho"][tb]
    assert not det["ambiguous"][ta] and not det["ambiguous"][tb]
    b = sc.bin_of(det["l"][ta], det["k"][ta], det["j"][ta])
    assert b == sc.bin_of(det["l"][tb], det["k"][tb], det["j"][tb])
    pcl, swapped = sc.ordered_bin_sums(det, lut, b, b_idx, a_idx)
    assert pcl != swapped
    assert got_row[b] == pcl


def _assert_batch(ko, kp, d, res, counts, lut, tie, label):
    assert list(np.diff(ko)) == [len(r["keypoints"]) for r in res]
    amb = tot = 0
    for s, r in enumerate(res):
        a, b = ko[s], ko[s + 1]
        assert list(r["n_neighbors"]) == [counts[s]]
        assert bits_equal(kp[a:b], r["keypoints"]) and bits_equal(d[a:b], r["descriptors"]), s
        ref = sc.reference_descriptors(r["cloud_full"], r["keypoints"], R)
        st = sc.check_descriptors_against_reference(r["cloud_full"], r["keypoints"], R, d[a:b], ref=ref)
        if tie[s] is not None:
            _assert_tie_order(ref, lut, d[a], *tie[s])
        amb, tot = amb + st["ambiguous"], tot + st["contributions"]
    assert amb <= 1e-3 * tot, (amb, tot)
    print("\n%s: %d scans, ambiguous share %.1e of %d contributions" % (label, len(res), amb / tot, tot))


# the pole of the list-capacity scans sits inside one row of the batch's surface grid, and so does their clutter
WPOLE_Y, WSLAB = -0.22, (-0.42, -0.02)


def _grid_row(y, P):
    """Row of the batch's surface grid (fe_api.cu surface_grid over the crop box, fe_kernels.cuh surf_cell) of y."""
    reach = F32((P.descriptor_radius * 1.2) * 1.001 + 1e-3)
    sy0 = F32(F32(P.y_min) - reach)
    inv = F32(1.0) / F32(P.descriptor_radius / 5.0 * 1.001)
    return np.floor((np.asarray(y, F32) - sy0) * inv).astype(np.int64)


def wcap_scans(ob, counts, seed):
    """Scans whose keypoint has all its `count` neighbours in ONE row of the surface grid: K4b's warp of that row lists
    them all, so 512 fills its list exactly (MARK_WCAP) and 513 overflows it (K4d then finds the neighbours itself)."""
    P = ob.node_default()
    wp = pole(1.0, WPOLE_Y)
    kp = ob.process_scan(P, wp, 0.0, 0.0, mode=1)["keypoints"][0]
    rng = np.random.default_rng(seed)
    scans = [np.concatenate([wp, clutter(rng, kp, n - len(wp), yslab=WSLAB)]) for n in counts]
    for s, n in zip(scans, counts):
        nb = s[sc.d2_f32(kp[:3], s[:, :3]) < sc.radius_sq_float(R)]
        assert len(nb) == n and len(set(_grid_row(nb[:, 1], P))) == 1
    return scans


def test_tier_ladder_through_a_large_batch(ob, pole_kp, lut):
    counts = [pole_kp[1] + 3] + LADDER + [300, 2000]           # 19 scans: warp kernel and batch instantiations
    pts, offs, rp, tie = ladder_scans(pole_kp, counts, 21)
    wc = wcap_scans(ob, [512, 513], 22)                       # and one warp at its list capacity, then one beyond
    pts = np.concatenate([pts] + wc)
    offs = np.concatenate([offs, offs[-1] + np.cumsum([len(s) for s in wc])]).astype(np.int64)
    rp = np.zeros((len(offs) - 1, 2))
    counts, tie = counts + [512, 513], tie + [None, None]
    res = _oracle_scans(ob, pts, offs)
    nd = _node(ob)
    ko, kp, d = nd.processBatch(pts, offs, rp)
    _assert_batch(ko, kp, d, res, counts, lut, tie, "batch of %d scans" % len(counts))
    assert nd.batchStats()["descriptors_unordered"] == 0
    nd.close()


def test_tier_ladder_through_small_calls_and_the_lean_chain(ob, pole_kp, lut):
    small = [pole_kp[1] + 3, 255, 256, 257, 511, 512, 513, 1535, 1536]   # the lean chain's first instantiations suffice
    large = [1537, 4095, 4096, 4097, 8191, 8192, 8193, 20000]       # keypoints for the larger instantiations
    nd = _node(ob)
    for counts, seed in ((small, 31), (large, 32)):
        pts, offs, rp, tie = ladder_scans(pole_kp, counts, seed)
        res = _oracle_scans(ob, pts, offs)
        before, replays = nd.leanReruns(), nd.enableGraphs(True)
        ko, kp, d = nd.processBatch(pts, offs, rp)         # block per keypoint, lean chain
        _assert_batch(ko, kp, d, res, counts, lut, tie, "call of %d scans" % len(counts))
        assert nd.leanReruns() == before + (1 if counts is large else 0)
        for rep in range(3):                               # a captured graph of the same shape, then its replays
            ko, kp, d = nd.processBatch(pts, offs, rp)
            _assert_batch(ko, kp, d, res, counts, lut, tie, "replay")
        assert nd.enableGraphs(True) > replays
        assert nd.leanReruns() == before + (1 if counts is large else 0)   # the lean chain stays off after a rerun
    nd.close()


def test_a_bin_with_more_than_8192_contributions_is_summed_order_free_and_stays_in_the_bound(ob, pole_kp):
    import torch
    kp, npole = pole_kp
    rng = np.random.default_rng(41)
    ax = sc.axis_draws(1)[0].astype(np.float64)
    alpha = np.rad2deg(np.arctan2(ax[1], ax[0]))
    l = int(((180.0 - alpha) % 360.0) // 30)                 # the azimuth bin pointing behind the crop box
    f0 = alpha + 30 * l
    block = clutter(rng, kp, 9000, box=((2.2, 2.45), (86.0, 94.0), (f0 + 6, f0 + 24)))
    dense = np.concatenate([pole(), block, clutter(rng, kp, 500)])
    others, offs_o, _, _ = ladder_scans(pole_kp, [600, 5000], 42)
    pts = np.concatenate([others[:offs_o[1]], dense, others[offs_o[1]:]])
    offs = np.array([0, offs_o[1], offs_o[1] + len(dense), len(pts)], np.int64)
    res = _oracle_scans(ob, pts, offs)
    nd = _node(ob)
    dp = torch.from_numpy(pts).cuda()
    ko, K, kp_ptr, d_ptr = nd.processBatchDevice(dp.data_ptr(), offs, np.zeros((3, 2)))
    d = nd.download(d_ptr, (K, sc.DESC_LEN))
    unordered = nd.batchStats()["descriptors_unordered"]
    assert unordered == 1
    assert list(ko) == [0, 1, 2, 3]
    assert bits_equal(d[0], res[0]["descriptors"][0]) and bits_equal(d[2], res[2]["descriptors"][0])
    ref = sc.reference_descriptors(res[1]["cloud_full"], res[1]["keypoints"], R)
    bn = int(np.argmax(ref["n"][0]))
    assert ref["n"][0, bn] > 8192 and bn == sc.bin_of(l, 5, 14)
    rest = np.arange(sc.DESC_LEN) != bn
    assert bits_equal(d[1, rest], res[1]["descriptors"][0, rest])
    sc.check_descriptors_against_reference(res[1]["cloud_full"], res[1]["keypoints"], R, d[1:2], ref=ref)
    print("\norder-free bin: descriptors_unordered %d, %d contributions in the bin, device %r, oracle %r"
          % (unordered, ref["n"][0, bn], d[1, bn], res[1]["descriptors"][0, bn]))
    nd.close()


def test_a_scan_of_2_20_points_is_processed_and_one_more_is_refused(ob, pole_kp, lut):
    """Two tie groups whose later member sits at a high index: with the order key's index field any narrower than 20
    bits, 2^19 + 5 would sort before 1000 and the sum would change; 2^20 - 1 is the largest index a scan can have."""
    from feature_extraction_b200 import FeatureExtractionError, _native
    kp, npole = pole_kp
    rng = np.random.default_rng(51)
    n = 1 << 20
    g1, g2 = sc.tie_group(kp, 180.0), sc.tie_group(kp, 140.0)
    assert all((g[k][:, 0] < 0).all() for g in (g1, g2) for k in g)
    scan = np.stack([rng.uniform(-70, -20, n), rng.uniform(-40, 40, n), rng.uniform(-1, 3, n), np.zeros(n)], 1).astype(F32)
    scan[:npole] = pole()
    scan[3000:6000] = clutter(rng, kp, 3000, groups=(180.0, 140.0))
    ties = []
    for g, (ib, ia) in ((g1, (1000, (1 << 19) + 5)), (g2, (2000, n - 1))):
        scan[ib], scan[ib + 1], scan[ia] = g["B"][0], g["C"][0], g["A"][0]
        scan[ib + 2:ib + 2 + len(g["extra"])] = g["extra"]
        ties.append((ib, ia))
    nd = _node(ob, max_points=n + 64, max_scans=4)
    over = np.concatenate([scan, scan[-2:-1]])
    with pytest.raises(FeatureExtractionError) as e:
        nd.processBatch(over, np.array([0, n + 1], np.int64), np.zeros((1, 2)))
    assert e.value.status == _native.FE_ERR_CAPACITY
    import torch
    d_over = torch.from_numpy(over).cuda()
    with pytest.raises(FeatureExtractionError) as e:
        nd.processBatchDevice(d_over.data_ptr(), np.array([0, n + 1], np.int64), np.zeros((1, 2)))
    assert e.value.status == _native.FE_ERR_CAPACITY
    del d_over
    r = ob.process_scan(ob.node_default(), scan, 0.0, 0.0, mode=1)
    assert len(r["keypoints"]) == 1 and r["n_neighbors"][0] == npole + 3000 + 6
    ko, kpg, d = nd.processBatch(scan, np.array([0, n], np.int64), np.zeros((1, 2)))
    assert bits_equal(kpg, r["keypoints"]) and bits_equal(d, r["descriptors"])
    ref = sc.reference_descriptors(r["cloud_full"], r["keypoints"], R)
    sc.check_descriptors_against_reference(r["cloud_full"], r["keypoints"], R, d, ref=ref)
    for ib, ia in ties:
        _assert_tie_order(ref, lut, d[0], ib, ia)
    # fe_estimate_descriptors: a cloud of 2^20 points is described the same; one more point is refused even when
    # nearly all of them are NaN
    de = nd.estimateDescriptors(r["cloud_full"], r["keypoints"])
    assert bits_equal(de, r["descriptors"])
    sparse = np.full((n + 1, 4), np.nan, F32)
    sparse[:8000] = r["cloud_full"][:8000]
    with pytest.raises(FeatureExtractionError) as e:
        nd.estimateDescriptors(sparse, r["keypoints"])
    assert e.value.status == _native.FE_ERR_CAPACITY
    assert bits_equal(nd.estimateDescriptors(sparse[:n], r["keypoints"]),
                      ob.estimate_descriptors(ob.node_default(), sparse[:n], r["keypoints"], mode=1)[0])
    nd.close()


def test_correctly_rounded_angles_stay_within_the_reference_bound(ob, synth):
    nd = _node(ob)
    nd.setAngleLibm(True)
    for cfg in (3, 4):
        pts, offs, rp = synth.generate(cfg, 2, scan_index_base=950)
        ko, kp, d = nd.processBatch(pts, offs, rp)
        for s in range(2):
            r = ob.process_scan(ob.node_default(), pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1)
            assert bits_equal(kp[ko[s]:ko[s + 1]], r["keypoints"])
            _check(r["cloud_full"], r["keypoints"], d[ko[s]:ko[s + 1]])
    nd.setAngleLibm(False)
    nd.close()
