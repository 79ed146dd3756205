"""An independent evaluation of the 3DSC descriptor (pcl::ShapeContext3DEstimation, PCL 1.8 conventions, as
include/fe_b200.h and DESIGN.md row H-N state them), plus the inputs the 3DSC tests build.  numpy and scipy only:
nothing here calls the oracle library, so a misreading of PCL that the oracle and the device share shows up here.

What the reference evaluates, per keypoint o and surface point q (float32 coordinates):

* Distance predicates, exact.  d2 = (dx*dx + dy*dy) + dz*dz in float32 of the float32 differences q - o.  q is a
  neighbour when d2 < (float)(R*R); the density of q counts the points p with d2(q, p) < (float)((R/5)^2), q itself
  included.  A neighbour with d2 < FLT_MIN (the keypoint itself) counts for support and for the RNG and contributes
  nothing.  The radial bin j is the first a in 1..15 with sqrtf(d2) <= radii[a] (j = a - 1), otherwise 0.  numpy's
  float32 operations are correctly rounded and never fused, so these decisions are the product's to the last bit.
* Tables.  radii[j] = (float)exp(log(R/10) + (j/15.f) * log(10)), theta[k] = k * (180.f/11), phi[l] = l * (360.f/12),
  all as PCL builds them.  Weights are V^(-1/3) / rho in float64, V = dphi * (cos theta_k - cos theta_k+1) *
  (r_j+1^3 - r_j^3) / 3 computed analytically from those float edges.
* Angles, float64.  theta = the angle between q - o and +z; phi = the counter-clockwise angle about +z from the
  keypoint's x axis to the horizontal part of q - o, in [0, 360).  Bin: the first edge >= the value (theta edges
  1..11, phi edges 1..12), otherwise bin 0; a neighbour with no horizontal offset lands in azimuth bin 0.
* Axes.  std::mt19937(12345) draws, each turned into a double by / 2^32 and then into a float; the axis is (u0, u1)
  normalised, the third draw is discarded.  Three draws per keypoint that is finite and has at least one neighbour, in
  keypoint order, from a fresh stream per estimateDescriptors call and per scan of a batch.

Where the product's angles go through libm the reference allows a band.  The product normalises q - o and its
horizontal projection in float (relative error a few 2^-24), evaluates atan2f / acosf to within 1 ulp and multiplies by
57.29578f (within 1e-8 of 180/pi); the float differences q - o are rounded once (2^-24 relative).  The elevation edges
used for binning (16.36 deg apart) are at least 16.36 deg from the poles, where acos's conditioning 1/sin(theta) is at
most 3.6, so theta is within about 2^-20 rad of the exact angle; the azimuth of a horizontal offset D_h of a distance D
is within about 2^-20 * D / D_h rad, and 360 - phi adds half an ulp of 360 deg (2^-21.9 rad).  One more term: PCL
projects the neighbour itself (q - lambda * normal, lambda = fl(q.z - o.z)) and subtracts the origin afterwards, so the
projection keeps a z residue of up to about 2^-24 * Z, Z = max(|o.z|, |q.z|), which tilts the azimuth near the 0 and 180
deg edges by up to 2^-24 * Z / D_h.  That is below 2^-17 * D / D_h while Z < 2^7 * D, true of every real scan tested (a
neighbour closer than Z / 128, 1.6 cm for a keypoint 2 m above the sensor); closer neighbours get the band scaled by Z / 128
instead of D.  A contribution is therefore called AMBIGUOUS
  - in theta when |theta - edge| < 2^-17 rad for an edge theta[1..10],
  - in phi when |phi - edge| < 2^-17 * max(D, Z / 128) / D_h rad for an edge phi[0..12] (0 and 360 deg both separate
    bin 11 from bin 0), and in every azimuth bin when D_h < 2^-10 * D,
which leaves a factor of 8 or more over the error analysis; the tolerance-boundary report's kinds 8 and 9 count the
same neighbourhoods.  An ambiguous contribution may land in any of its candidate bins, with that bin's weight.

The check (check_descriptors_against_reference) per bin: lo - tol <= got <= hi + tol, lo the sum of the sure
contributions, hi that plus every ambiguous contribution that could land in the bin, and
  tol = ((n_b + 4) * 2^-24 + 2e-6) * hi,
n_b the bin's contribution count: the sequential float sum of n_b terms, each weight fl(fl(1/rho) * lut) two roundings
off, plus the float32 volume table (powf(V, 1/3.f), cosf of float radians, float cubes) within 2e-6 of V^(-1/3).  The
row's total mass is held to the sum of the bins' bounds.  Measured against the CPU oracle on configs 1-4 at R = 2.5
and 5 and on config 2 at R = 0.3 and 6 (tests/test_oracle_sc3d.py prints it), the largest deviation of an unambiguous
bin stays below 0.18 of its tolerance; the float32 volume table is within 3.3e-7 of V^(-1/3) at those radii.
"""
import numpy as np
from scipy.spatial import cKDTree

DESC_LEN, NL, NK, NJ = 1980, 12, 11, 15
F32 = np.float32
FLT_MIN = float(np.finfo(np.float32).tiny)
DEG = np.pi / 180.0
BAND = 2.0 ** -17      # rad
POLE = 2.0 ** -10      # D_h / D below which the azimuth is anyone's
SEED = 12345


# ---------------------------------------------------------------------------------------------------------------
# tables
# ---------------------------------------------------------------------------------------------------------------
def radius_sq_float(r):
    """(float)(r * r) with r a double: how every radius predicate narrows its radius."""
    return F32(float(r) * float(r))


def tables(R):
    """(radii[16], theta[12], phi[13]) float32 in PCL's formula, and w[11, 15] = V^(-1/3) float64 per (k, j)."""
    R = float(R)
    rmin = R / 10.0
    radii = np.array([F32(np.exp(np.log(rmin) + float(F32(j) / F32(NJ)) * np.log(R / rmin))) for j in range(NJ + 1)], F32)
    theta = np.array([F32(k) * (F32(180.0) / F32(NK)) for k in range(NK + 1)], F32)
    phi = np.array([F32(l) * (F32(360.0) / F32(NL)) for l in range(NL + 1)], F32)
    r = radii.astype(np.float64)
    t = theta.astype(np.float64) * DEG
    dphi = float(phi[1] - phi[0]) * DEG
    V = dphi * (np.cos(t[:-1]) - np.cos(t[1:]))[:, None] * ((r[1:] ** 3 - r[:-1] ** 3) / 3.0)[None, :]
    return radii, theta, phi, V ** (-1.0 / 3.0)


def axis_draws(n_axes):
    """(n_axes, 2) float32 (u0, u1): std::mt19937(12345) through numpy's legacy seeding (the same stream), three draws
    per axis, the third discarded."""
    raw = np.random.RandomState(SEED).randint(0, 2 ** 32, size=3 * max(n_axes, 1), dtype=np.uint64)
    u = (raw.astype(np.float64) / 4294967296.0).astype(F32)
    return u.reshape(-1, 3)[:n_axes, :2]


def mt19937_raw(n):
    return np.random.RandomState(SEED).randint(0, 2 ** 32, size=n, dtype=np.uint64)


# ---------------------------------------------------------------------------------------------------------------
# exact float32 neighbourhoods
# ---------------------------------------------------------------------------------------------------------------
def d2_f32(o, q):
    """FLANN L2_Simple in float32: (dx*dx + dy*dy) + dz*dz of float32 differences; o (3,) or (n, 3), q (n, 3)."""
    o = np.asarray(o, F32)
    q = np.asarray(q, F32)
    dx, dy, dz = (q[..., 0] - o[..., 0]), (q[..., 1] - o[..., 1]), (q[..., 2] - o[..., 2])
    return (dx * dx + dy * dy) + dz * dz


class Cloud:
    """The finite points of a cloud with a KD-tree for candidates; every decision is the exact float32 predicate."""

    def __init__(self, cloud):
        c = np.asarray(cloud, F32)[:, :3]
        fin = np.isfinite(c).all(axis=1)
        self.idx = np.nonzero(fin)[0]
        self.xyz = np.ascontiguousarray(c[fin])
        self.tree = cKDTree(self.xyz.astype(np.float64)) if len(self.xyz) else None

    def within(self, o, r2f):
        """indices into the original cloud of the points p with d2(o, p) < r2f, and their d2."""
        if self.tree is None:
            return np.zeros(0, np.int64), np.zeros(0, F32)
        cand = np.asarray(self.tree.query_ball_point(np.asarray(o, np.float64), np.sqrt(float(r2f)) * (1 + 1e-5) + 1e-30),
                          np.int64)
        if len(cand) == 0:
            return np.zeros(0, np.int64), np.zeros(0, F32)
        d2 = d2_f32(np.asarray(o, F32)[:3], self.xyz[cand])
        m = d2 < r2f
        return self.idx[cand[m]], d2[m]

    def counts(self, pts, r2f):
        """for every point of pts, the number of cloud points p with d2(pt, p) < r2f (exact)."""
        pts = np.asarray(pts, F32)[:, :3]
        if self.tree is None or len(pts) == 0:
            return np.zeros(len(pts), np.int64)
        r = np.sqrt(float(r2f))
        p64 = pts.astype(np.float64)
        lo = self.tree.query_ball_point(p64, r * (1 - 1e-5), return_length=True)
        hi = self.tree.query_ball_point(p64, r * (1 + 1e-5) + 1e-30, return_length=True)
        out = np.asarray(hi, np.int64).copy()
        for i in np.nonzero(np.asarray(lo) != np.asarray(hi))[0]:   # a point near the sphere: decide exactly
            cand = np.asarray(self.tree.query_ball_point(p64[i], r * (1 + 1e-5) + 1e-30), np.int64)
            out[i] = int((d2_f32(pts[i], self.xyz[cand]) < r2f).sum())
        return out


# ---------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------
def _angle_candidates(v, edges, band, wrap):
    """Bins a value v (rad) may take given edges (rad) 0..n and a band per value.  Nominal: the first edge a >= 1 with
    v <= edge -> a - 1, otherwise 0.  Returns (nominal (m,), cand list of arrays)."""
    n = len(edges) - 1
    nominal = np.zeros(len(v), np.int64)
    done = np.zeros(len(v), bool)
    for a in range(1, n + 1):
        hit = ~done & (v <= edges[a])
        nominal[hit] = a - 1
        done |= hit
    cands = [{int(x)} for x in nominal]
    lo_a, hi_a = (0, n) if wrap else (1, n - 1)
    for a in range(lo_a, hi_a + 1):
        near = np.nonzero(np.abs(v - edges[a]) < band)[0]
        pair = (n - 1, 0) if a in (0, n) else (a - 1, a)
        for i in near:
            cands[i].update(pair)
    return nominal, cands


def reference_descriptors(cloud, keypoints, R, axis_offset=0):
    """-> dict with, per keypoint, `nan` (bool), `lo`, `hi` (1980 float64), `n` (contributions per bin, int),
    `ambiguous` (contributions with more than one candidate bin), `contrib` (contributions), `n_neighbors`, `mass_lo`
    and `mass_hi` (bounds of the row's total), `detail` (None, or for every contribution its cloud index, nominal
    (l, k, j), d2, density and whether it is ambiguous), and `axes_used`, the axes drawn.  axis_offset: axes already drawn before
    these keypoints (0 for a fresh call)."""
    cl = Cloud(cloud)
    cfull = np.asarray(cloud, F32)
    kps = np.asarray(keypoints, F32)
    radii, theta, phi, wvol = tables(R)
    R2f = radius_sq_float(R)
    rho2f = radius_sq_float(R / 5.0)
    th_e = theta.astype(np.float64) * DEG
    ph_e = phi.astype(np.float64) * DEG
    K = len(kps)
    out = {"nan": np.zeros(K, bool), "lo": np.zeros((K, DESC_LEN)), "hi": np.zeros((K, DESC_LEN)),
           "n": np.zeros((K, DESC_LEN), np.int64), "ambiguous": np.zeros(K, np.int64), "contrib": np.zeros(K, np.int64),
           "n_neighbors": np.zeros(K, np.int64), "mass_lo": np.zeros(K), "mass_hi": np.zeros(K), "detail": [None] * K}
    nbrs = []
    for i in range(K):
        o = kps[i, :3]
        if not np.isfinite(o).all():
            nbrs.append(None)
            continue
        idx, d2 = cl.within(o, R2f)
        nbrs.append((idx, d2))
        out["n_neighbors"][i] = len(idx)
    ranked = [i for i in range(K) if nbrs[i] is not None and len(nbrs[i][0]) > 0]
    axes = axis_draws(axis_offset + len(ranked))[axis_offset:]
    out["axes_used"] = len(ranked)
    rank = {g: r for r, g in enumerate(ranked)}
    for i in range(K):
        if i not in rank:
            out["nan"][i] = True
            continue
        idx, d2 = nbrs[i]
        keep = d2 >= F32(FLT_MIN)
        idx, d2 = idx[keep], d2[keep]
        if len(idx) == 0:
            continue
        q = cfull[idx, :3]
        rho = cl.counts(q, rho2f)
        ok = rho > 0
        idx, d2, q, rho = idx[ok], d2[ok], q[ok], rho[ok]
        rr = np.sqrt(d2)                                   # float32 sqrt, correctly rounded
        j = np.zeros(len(rr), np.int64)
        jd = np.zeros(len(rr), bool)
        for a in range(1, NJ + 1):
            hit = ~jd & (rr <= radii[a])
            j[hit] = a - 1
            jd |= hit
        o = kps[i, :3].astype(np.float64)
        v = q.astype(np.float64) - o                        # exact
        D = np.sqrt((v * v).sum(axis=1))
        Dh = np.hypot(v[:, 0], v[:, 1])
        th = np.arctan2(Dh, v[:, 2])                        # [0, pi]
        k, kc = _angle_candidates(th, th_e, BAND, wrap=False)
        ax = axes[rank[i]].astype(np.float64)
        ph = np.mod(np.arctan2(ax[0] * v[:, 1] - ax[1] * v[:, 0], ax[0] * v[:, 0] + ax[1] * v[:, 1]), 2 * np.pi)
        ph = np.where(Dh == 0, 0.0, ph)
        with np.errstate(divide="ignore"):
            Z = np.maximum(abs(float(kps[i, 2])), np.abs(q[:, 2].astype(np.float64)))
            band = np.where(Dh > 0, BAND * np.maximum(D, Z / 128.0) / np.maximum(Dh, 1e-300), np.inf)
        n_ph = len(ph_e) - 1
        l_nom = np.zeros(len(ph), np.int64)
        ld = np.zeros(len(ph), bool)
        for a in range(1, n_ph + 1):
            hit = ~ld & (ph <= ph_e[a]) & (Dh > 0)
            l_nom[hit] = a - 1
            ld |= hit
        lc = [{int(x)} for x in l_nom]
        for a in range(0, n_ph + 1):
            near = np.nonzero(np.abs(ph - ph_e[a]) < band)[0]
            pair = (n_ph - 1, 0) if a in (0, n_ph) else (a - 1, a)
            for t in near:
                lc[t].update(pair)
        for t in np.nonzero(Dh < POLE * D)[0]:
            lc[t] = set(range(NL))
        inv_rho = 1.0 / rho.astype(np.float64)
        lo, hi, n = out["lo"][i], out["hi"][i], out["n"][i]
        amb = 0
        mlo = mhi = 0.0
        for t in range(len(rr)):
            ks, ls = kc[t], lc[t]
            ws = [wvol[kk, j[t]] * inv_rho[t] for kk in ks]
            if len(ks) == 1 and len(ls) == 1:
                b = l_nom[t] * 165 + k[t] * 15 + j[t]
                lo[b] += ws[0]
                hi[b] += ws[0]
                n[b] += 1
            else:
                amb += 1
                for kk, w in zip(ks, ws):
                    for ll in ls:
                        b = ll * 165 + kk * 15 + j[t]
                        hi[b] += w
                        n[b] += 1
            mlo += min(ws)
            mhi += max(ws)
        out["ambiguous"][i] = amb
        out["detail"][i] = {"idx": idx, "l": l_nom, "k": k, "j": j, "d2": d2, "rho": rho,
                            "ambiguous": np.array([len(kc[t]) * len(lc[t]) > 1 for t in range(len(rr))], bool)}
        out["contrib"][i] = len(rr)
        out["mass_lo"][i] = mlo
        out["mass_hi"][i] = mhi
    return out


def tolerance(hi, n):
    return ((n + 4) * 2.0 ** -24 + 2e-6) * hi


def check_descriptors_against_reference(cloud, keypoints, R, got, axis_offset=0, ref=None):
    """Assert that `got` (K, 1980) float32 are the 3DSC rows of `keypoints` in `cloud` at radius R within the bound
    above.  -> dict(rows, unambiguous_rows, ambiguous, contributions, worst): worst is the largest deviation of an
    unambiguous bin from the reference relative to its tolerance."""
    if ref is None:
        ref = reference_descriptors(cloud, keypoints, R, axis_offset)
    got = np.asarray(got, np.float32)
    K = len(ref["nan"])
    assert got.shape == (K, DESC_LEN), got.shape
    g_nan = np.isnan(got).all(axis=1)
    assert not np.isnan(got[~g_nan]).any(), "a row is partly NaN"
    bad = np.nonzero(g_nan != ref["nan"])[0]
    assert len(bad) == 0, "NaN rows differ from the reference at keypoints %s" % bad[:10]
    worst = 0.0
    g64 = got.astype(np.float64)
    for i in np.nonzero(~ref["nan"])[0]:
        lo, hi, n = ref["lo"][i], ref["hi"][i], ref["n"][i]
        tol = tolerance(hi, n)
        g = g64[i]
        over = np.nonzero((g < lo - tol) | (g > hi + tol))[0]
        assert len(over) == 0, ("keypoint %d: bins %s outside the reference: got %s, lo %s, hi %s, contributions %s"
                                % (i, over[:8], g[over[:8]], lo[over[:8]], hi[over[:8]], n[over[:8]]))
        exact = (lo == hi) & (hi > 0)
        if exact.any():
            worst = max(worst, float((np.abs(g[exact] - hi[exact]) / tol[exact]).max()))
        tot_tol = tol.sum()
        s = g.sum()
        assert ref["mass_lo"][i] - tot_tol <= s <= ref["mass_hi"][i] + tot_tol, \
            "keypoint %d: total mass %r outside [%r, %r] +- %r" % (i, s, ref["mass_lo"][i], ref["mass_hi"][i], tot_tol)
    rows = int((~ref["nan"]).sum())
    return {"rows": rows, "unambiguous_rows": int(((ref["ambiguous"] == 0) & ~ref["nan"]).sum()),
            "ambiguous": int(ref["ambiguous"].sum()), "contributions": int(ref["contrib"].sum()), "worst": worst}


# ---------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------
def float_with_sqrt_square(target, want):
    """A float32 c near `target` with sqrt(fl(c*c)) == want exactly (want a float32), or None."""
    c = F32(target)
    for _ in range(64):
        s = np.sqrt(c * c)
        if s == want:
            return c
        c = np.nextafter(c, F32(np.inf) if s < want else F32(-np.inf))
    return None


def float_with_square(target, want_sq):
    """A float32 c near `target` with fl(c*c) == want_sq, or None."""
    c = F32(target)
    for _ in range(64):
        s = c * c
        if s == want_sq:
            return c
        c = np.nextafter(c, F32(np.inf) if s < want_sq else F32(-np.inf))
    return None


def float_around_square(target_sq):
    """(c_in, c_out): the largest float32 c with fl(c*c) < target_sq and the next one up (fl(c*c) >= target_sq)."""
    c = np.sqrt(F32(target_sq))
    while c * c >= target_sq:
        c = np.nextafter(c, F32(0))
    while np.nextafter(c, F32(np.inf)) ** 2 < target_sq:
        c = np.nextafter(c, F32(np.inf))
    return c, np.nextafter(c, F32(np.inf))


def ball_points(rng, center, n, r_lo, r_hi):
    """n float32 points uniform in the shell r_lo <= |p - center| <= r_hi (float64 radii; callers keep a margin from
    the float predicates they care about)."""
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    r = (r_lo ** 3 + rng.random(n) * (r_hi ** 3 - r_lo ** 3)) ** (1.0 / 3.0)
    p = np.asarray(center, np.float64)[:3] + u * r[:, None]
    return p.astype(F32)


def with_count(rng, center, R, count, lo_frac=0.12, hi_frac=0.98):
    """Exactly `count` points whose float d2 to `center` is below (float)(R^2), spread through the shell
    [lo_frac R, hi_frac R] (every radial bin but the first few, every angle), as (count, 4) float32 with w = 0."""
    if count == 0:
        return np.zeros((0, 4), F32)
    p = ball_points(rng, center, count, lo_frac * R, hi_frac * R)
    assert (d2_f32(np.asarray(center, F32)[:3], p) < radius_sq_float(R)).all()
    return np.concatenate([p, np.zeros((count, 1), F32)], axis=1)


def ordered_bin_sums(detail, lut, b, first, second):
    """The float32 sum of bin b as PCL forms it, weights fl(fl(1/rho) * lut[b]) added in ascending (d2, index) order,
    and the same sum with the contributions of cloud indices `first` and `second` (a d2 tie) in each other's places.
    -> (in order, swapped).  A test whose two sums are equal cannot see the order."""
    sel = np.nonzero(detail["l"] * 165 + detail["k"] * 15 + detail["j"] == b)[0]
    order = sel[np.lexsort((detail["idx"][sel], detail["d2"][sel]))]
    idx = list(detail["idx"][order])
    w = [F32(F32(1) / F32(r)) * F32(lut[b]) for r in detail["rho"][order]]
    ia, ib = idx.index(first), idx.index(second)
    sw = list(w)
    sw[ia], sw[ib] = w[ib], w[ia]
    acc, acc_s = F32(0), F32(0)
    for x, y in zip(w, sw):
        acc, acc_s = F32(acc + x), F32(acc_s + y)
    return acc, acc_s


def tie_group(kp, ang_deg):
    """Contributions that make the (d2, index) order visible, placed at azimuth ang_deg (about +x) from keypoint kp:
    C, then B and A at the same float d2 (mirrored in z about kp), all three in one bin, and twelve points beyond R = 2.5
    within R/5 of A only, so that A's density (15) differs from B's and C's (3).  -> dict of (n, 4) float32 arrays
    "C", "B", "A", "extra"; B must come before A in the cloud."""
    c, s = np.cos(np.deg2rad(ang_deg)), np.sin(np.deg2rad(ang_deg))
    o = np.asarray(kp, np.float64)[:3]

    def at(rel):
        rel = np.asarray(rel, np.float64).reshape(-1, 3)
        p = np.stack([o[0] + c * rel[:, 0] - s * rel[:, 1], o[1] + s * rel[:, 0] + c * rel[:, 1], o[2] + rel[:, 2]], 1)
        return np.concatenate([p.astype(F32), np.zeros((len(p), 1), F32)], 1)

    a = at([2.3, 0.2, 0.01])
    b = a.copy()
    b[0, 2] = F32(F32(kp[2]) - (a[0, 2] - F32(kp[2])))     # the mirror image in float, then nudged onto the same d2
    want = d2_f32(np.asarray(kp, F32)[:3], a[:, :3])[0]
    for _ in range(64):
        d = d2_f32(np.asarray(kp, F32)[:3], b[:, :3])[0]
        if d == want:
            break
        b[0, 2] = np.nextafter(b[0, 2], F32(-np.inf) if (d < want) == (b[0, 2] < kp[2]) else F32(np.inf))
    assert d2_f32(np.asarray(kp, F32)[:3], b[:, :3])[0] == want
    extra = at([(2.46, 0.17, 0.47), (2.46, 0.2, 0.47), (2.46, 0.23, 0.47), (2.48, 0.17, 0.47), (2.48, 0.2, 0.47),
                (2.48, 0.23, 0.47), (2.46, 0.17, 0.475), (2.46, 0.2, 0.475), (2.46, 0.23, 0.475), (2.48, 0.2, 0.475),
                (2.46, 0.17, 0.48), (2.46, 0.2, 0.48)])
    return {"C": at([2.25, 0.2, 0.0]), "B": b, "A": a, "extra": extra}


def bin_of(l, k, j):
    return l * 165 + k * 15 + j
