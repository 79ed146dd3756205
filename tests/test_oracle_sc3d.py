"""The CPU oracle's 3DSC descriptors against the independent float64 evaluation of sc3d_cases.py: first the reference
on constructed neighbourhoods whose bins are known by construction, then the oracle against the reference on those
and on real scans."""
import numpy as np
import pytest

import sc3d_cases as sc

F32 = np.float32


def _params(ob, R):
    P = ob.node_default()
    P.descriptor_radius = R
    return P


def test_tables_and_axis_stream_are_pcls(ob):
    for R in (0.3, 1.0, 2.5, 5.0, 6.0, 7.3):
        radii, theta, phi, lut = ob.sc3d_tables(R)
        r, t, p, w = sc.tables(R)
        for a, b in ((radii, r), (theta, t), (phi, p)):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), R
        # the float32 volume table against the analytic V^(-1/3), every azimuth block the same
        L = lut.astype(np.float64).reshape(12, 11, 15)
        assert np.array_equal(L, np.broadcast_to(L[0], L.shape))
        assert np.abs(L[0] / w - 1).max() < 2e-6, R
    raw, f = ob.mt19937_draws(12345, 3 * 70000)
    assert np.array_equal(raw.astype(np.uint64), sc.mt19937_raw(3 * 70000))
    assert np.array_equal(f.reshape(-1, 3)[:, :2].view(np.uint32), sc.axis_draws(70000).view(np.uint32))


def edge_cloud(R):
    """Keypoint at the origin and neighbours placed on and around every decision of the binning.  -> (cloud (n, 4),
    expected {cloud index: (l or None, k or None, j or None)} for the neighbours whose bin is known by construction,
    excluded cloud indices)."""
    radii, theta, phi, _ = sc.tables(R)
    R2f = sc.radius_sq_float(R)
    ax = sc.axis_draws(1)[0].astype(np.float64)
    alpha = np.arctan2(ax[1], ax[0])
    pts, expect, excluded, poles = [], {}, [], []

    def add(p, e=None):
        pts.append([F32(p[0]), F32(p[1]), F32(p[2]), F32(0)])
        if e is not None:
            expect[len(pts) - 1] = e

    add((0, 0, 0))                                           # the keypoint itself: support and RNG, no contribution
    for a in range(1, 15):                                   # every radial edge: on it, one float inside and outside
        c = sc.float_with_sqrt_square(radii[a], radii[a])
        assert c is not None, a
        add((c, 0, 0), (None, 5, a - 1))
        cin = sc.float_with_sqrt_square(np.nextafter(radii[a], F32(0)), np.nextafter(radii[a], F32(0)))
        add((0, cin, 0), (None, 5, a - 1))
        cout = sc.float_with_sqrt_square(np.nextafter(radii[a], F32(9)), np.nextafter(radii[a], F32(9)))
        add((-cout, 0, 0), (None, 5, a))
    c_in, c_out = sc.float_around_square(R2f)               # the last float inside the sphere and the first outside
    add((0, -c_out, 0))
    excluded.append(len(pts) - 1)
    c_on = sc.float_with_square(R, R2f)                      # d2 == (float)R^2 exactly, where R^2 is a float square
    if c_on is not None:
        add((-c_on, -0.0, 0))
        excluded.append(len(pts) - 1)
    add((0, -c_in, 0))
    r_in = np.sqrt(c_in * c_in)                              # beyond radii[15] PCL's loop finds no shell: bin 0
    expect[len(pts) - 1] = (None, 5, 14 if r_in <= radii[15] else 0)
    add((F32(R / 25), F32(R / 50), F32(R / 100)), (None, None, 0))   # r < R/10: the first shell
    add((0, 0, F32(R * 0.4)), (0, 0, None))                  # straight above: no azimuth, bin 0
    add((0, 0, F32(-R * 0.45)), (0, 10, None))               # straight below
    poles += [len(pts) - 2, len(pts) - 1]
    d = 2e-4                                                 # rad, far beyond the band at these distances
    for a in range(12):                                      # both sides of every azimuth edge, at 73 deg elevation
        for s, l in ((-1, (a - 1) % 12), (1, a)):
            ang = alpha + np.deg2rad(30.0 * a) + s * d
            add((0.6 * R * np.cos(ang), 0.6 * R * np.sin(ang), 0.18 * R), (l, 4, None))
    for a in range(1, 11):                                   # both sides of every elevation edge
        for s, k in ((-1, a - 1), (1, a)):
            t = np.deg2rad(float(theta[a])) + s * d
            ang = alpha + np.deg2rad(15.0)
            add((0.7 * R * np.sin(t) * np.cos(ang), 0.7 * R * np.sin(t) * np.sin(ang), 0.7 * R * np.cos(t)), (0, k, None))
    return np.array(pts, F32), expect, excluded, poles


@pytest.mark.parametrize("R", [2.5, 0.3, 6.0])
def test_reference_bins_constructed_neighbours_as_built_and_the_oracle_agrees(ob, R):
    cloud, expect, excluded, poles = edge_cloud(R)
    kp = np.zeros((1, 4), F32)
    ref = sc.reference_descriptors(cloud, kp, R)
    det = ref["detail"][0]
    where = {int(i): t for t, i in enumerate(det["idx"])}
    assert 0 not in where                                    # the keypoint itself contributes nothing ...
    assert ref["n_neighbors"][0] == len(cloud) - len(excluded)   # ... but is a neighbour
    for i in excluded:
        assert i not in where
    for i, (l, k, j) in expect.items():
        t = where[i]
        got = (int(det["l"][t]), int(det["k"][t]), int(det["j"][t]))
        for want, g in zip((l, k, j), got):
            assert want is None or want == g, (i, (l, k, j), got)
        if i in poles:
            assert det["ambiguous"][t]                       # no horizontal offset: every azimuth bin is possible
        else:
            assert not det["ambiguous"][t], (i, got)
    d, _, nn = ob.estimate_descriptors(_params(ob, R), cloud, kp)
    assert nn[0] == ref["n_neighbors"][0]
    st = sc.check_descriptors_against_reference(cloud, kp, R, d, ref=ref)
    assert st["ambiguous"] == 2
    # the oracle follows PCL's arithmetic for a zero horizontal offset (a NaN azimuth): bin 0, as the reference says
    for i in poles:
        t = where[i]
        b = sc.bin_of(0, int(det["k"][t]), int(det["j"][t]))
        assert d[0, b] > 0


def tie_cloud():
    """Three contributions to one bin, two of them at the same d2 (mirrored in z about the keypoint's 90 deg elevation
    band) with different densities: points beyond R raise one of them.  The float sum depends on the (d2, index)
    order.  -> cloud, keypoints (one keypoint at the origin), the cloud indices of (C, first tie, second tie)."""
    pts = [[3.0, 0.0, 0.0],      # an unrelated neighbour first
           [2.3, 0.2, -0.01],    # B: tie, lower index
           [2.3, 0.2, 0.01],     # A: tie, higher index, extra density below
           [2.25, 0.2, 0.0],     # C: smaller d2, same bin
           [0.3, -1.0, 0.4]]
    # twelve points beyond R = 2.5 within R/5 of A only: densities 3, 3, 15 make the two orders round differently
    pts += [[x, y, z] for x, y, z in ((2.46, 0.17, 0.47), (2.46, 0.2, 0.47), (2.46, 0.23, 0.47), (2.48, 0.17, 0.47),
                                      (2.48, 0.2, 0.47), (2.48, 0.23, 0.47), (2.46, 0.17, 0.475), (2.46, 0.2, 0.475),
                                      (2.46, 0.23, 0.475), (2.48, 0.2, 0.475), (2.46, 0.17, 0.48), (2.46, 0.2, 0.48))]
    return np.array([p + [0.0] for p in pts], F32), np.zeros((1, 4), F32), (3, 1, 2)


def test_tied_squared_distances_are_summed_in_index_order(ob):
    R = 2.5
    cloud, kp, (c, b, a) = tie_cloud()
    d2 = sc.d2_f32(kp[0, :3], cloud[:, :3])
    assert d2[a] == d2[b] and d2[c] < d2[b] < sc.radius_sq_float(R)
    ref = sc.reference_descriptors(cloud, kp, R)
    det = ref["detail"][0]
    where = {int(i): t for t, i in enumerate(det["idx"])}
    bins = {sc.bin_of(det["l"][where[i]], det["k"][where[i]], det["j"][where[i]]) for i in (a, b, c)}
    assert len(bins) == 1 and not det["ambiguous"].any()
    rho = sc.Cloud(cloud).counts(cloud[[c, b, a], :3], sc.radius_sq_float(R / 5))
    assert rho[1] != rho[2]
    # the bin's float32 sum in (d2, index) order differs from the other order, so the order is observable
    lut = ob.sc3d_tables(R)[3]
    (bn,) = bins
    w = [F32(F32(1) / F32(r)) * lut[bn] for r in rho]
    pcl = (F32(0) + w[0] + w[1]) + w[2]
    swapped = (F32(0) + w[0] + w[2]) + w[1]
    assert pcl != swapped
    d, _, _ = ob.estimate_descriptors(_params(ob, R), cloud, kp)
    assert d[0, bn] == pcl
    sc.check_descriptors_against_reference(cloud, kp, R, d, ref=ref)


def rng_cloud(rng):
    """Keypoints that do and do not draw an axis, interleaved: NaN, no neighbour, only itself as neighbour, real
    neighbourhoods.  -> cloud, keypoints, rows expected NaN, rows expected all zeros."""
    cloud = np.concatenate([sc.with_count(rng, (20.0, 0.0, 0.0), 2.5, 300),
                            np.array([[50.0, 50.0, 0.0, 0.0]], F32),
                            sc.with_count(rng, (-20.0, 5.0, 0.5), 2.5, 300),
                            sc.with_count(rng, (0.0, -30.0, 1.0), 2.5, 200)])
    kps = np.array([[np.nan, 0, 0, 0], [90, 90, 0, 0], [50, 50, 0, 0], [20, 0, 0, 0], [0, 90, 0, 0],
                    [-20, 5, 0.5, 0], [50, 50, 0, 0], [0, -30, 1, 0], [np.inf, 1, 1, 0]], F32)
    return cloud, kps, [0, 1, 4, 8], [2, 6]


def test_only_keypoints_with_neighbours_draw_axes(ob):
    R = 2.5
    cloud, kps, nan_rows, zero_rows = rng_cloud(np.random.default_rng(7))
    ref = sc.reference_descriptors(cloud, kps, R)
    assert list(np.nonzero(ref["nan"])[0]) == nan_rows
    assert ref["axes_used"] == len(kps) - len(nan_rows)
    d, _, nn = ob.estimate_descriptors(_params(ob, R), cloud, kps)
    assert np.array_equal(nn, ref["n_neighbors"])
    assert np.isnan(d[nan_rows]).all() and (d[zero_rows] == 0).all()
    st = sc.check_descriptors_against_reference(cloud, kps, R, d, ref=ref)
    assert st["unambiguous_rows"] == st["rows"]
    # drawing for every keypoint instead would rotate the real rows' azimuth blocks out of the bound
    other = sc.reference_descriptors(cloud, kps[[0, 3, 5, 7]], R, axis_offset=1)
    with pytest.raises(AssertionError):
        sc.check_descriptors_against_reference(cloud, kps[[0, 3, 5, 7]], R, d[[0, 3, 5, 7]], ref=other)


SCAN_CASES = [(1, 2.5), (1, 5.0), (2, 2.5), (2, 5.0), (2, 0.3), (2, 6.0), (3, 2.5), (3, 5.0), (4, 2.5), (4, 5.0)]
MIN_UNAMBIGUOUS = {1: 0.6, 2: 0.6, 3: 0.5, 4: 0.7}   # share of checked rows without any ambiguous contribution


@pytest.fixture(scope="module")
def scan_totals():
    tot = {"rows": 0, "ambiguous": 0, "contributions": 0}
    yield tot
    assert tot["contributions"] > 0
    assert tot["ambiguous"] / tot["contributions"] < 1e-3, tot


@pytest.mark.parametrize("cfg,R", SCAN_CASES)
def test_oracle_descriptors_of_real_scans_are_within_the_reference_bound(ob, synth, cfg, R, scan_totals, capsys):
    pts, offs, rp = synth.generate(cfg, 3, scan_index_base=900)
    P = _params(ob, R)
    agg = {"rows": 0, "unambiguous_rows": 0, "ambiguous": 0, "contributions": 0, "worst": 0.0}
    for s in range(3):
        r = ob.process_scan(P, pts[offs[s]:offs[s + 1]], rp[s, 0], rp[s, 1], mode=1)
        st = sc.check_descriptors_against_reference(r["cloud_full"], r["keypoints"], R, r["descriptors"])
        for k in agg:
            agg[k] = max(agg[k], st[k]) if k == "worst" else agg[k] + st[k]
    assert agg["rows"] > 0
    assert agg["unambiguous_rows"] >= MIN_UNAMBIGUOUS[cfg] * agg["rows"], agg
    assert agg["ambiguous"] <= 1e-2 * agg["contributions"], agg
    assert agg["worst"] < 1.0
    for k in scan_totals:
        scan_totals[k] += agg[k]
    with capsys.disabled():
        print("\n3DSC oracle vs reference: config %d R %.1f: %d rows checked, %d unambiguous, ambiguous share %.1e of %d "
              "contributions, largest deviation %.3f of the bound"
              % (cfg, R, agg["rows"], agg["unambiguous_rows"], agg["ambiguous"] / max(agg["contributions"], 1),
                 agg["contributions"], agg["worst"]))
