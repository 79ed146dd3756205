"""Inputs and an independent float64 evaluation for the descriptor-matching tests (fe_match_descriptors)."""
import numpy as np

L, BLK, DESC_LEN, RECORD_FLOATS = 12, 165, 1980, 1996


def numpy_shift_distances(q, r):
    """(nq, nr, 12) float64: sum over l, m of (q[l, m] - r[(l + s) % 12, m])^2, from float64 copies."""
    A = np.asarray(q, np.float64).reshape(len(q), L, BLK)
    B = np.asarray(r, np.float64).reshape(len(r), L, BLK)
    out = np.empty((len(q), len(r), L))
    for s in range(L):
        Bs = np.roll(B, -s, axis=1)  # Bs[:, l] = B[:, (l + s) % 12]
        diff = A[:, None] - Bs[None]
        out[:, :, s] = np.einsum("ijlm,ijlm->ij", diff, diff)
    return out


def rolled(row, s):
    """A row whose block (l + s) mod 12 is block l of `row`: d_s(row, rolled(row, s)) == 0."""
    return np.roll(np.asarray(row, np.float32).reshape(L, BLK), s, axis=0).reshape(-1)


def random_rows(rng, n):
    return rng.random((n, DESC_LEN), dtype=np.float32) * rng.random((n, 1), dtype=np.float32)


def to_records(d):
    """(K, 1980) bins -> (K, 1996) records with the bins at offset 5 and something else around them."""
    rec = np.full((len(d), RECORD_FLOATS), -7.0, np.float32)
    rec[:, 5:5 + DESC_LEN] = d
    return rec


def constructed(rng):
    """(query, ref, query_offsets, ref_offsets): rolled copies, a duplicated reference row, NaN rows on both sides,
    empty groups on either side, and groups that do not start at row 0."""
    q = random_rows(rng, 14)
    r = random_rows(rng, 24)
    # group 0: q0..q3 vs r0..r7; q1 rolled by 5 into r3, q2's rolled copy in r6 and duplicated in r7 (second == best)
    r[3] = rolled(q[1], 5)
    r[6] = rolled(q[2], 11)
    r[7] = r[6]
    q[3] = np.nan  # a zero-neighbour keypoint: never matched
    # group 1: q4..q5 vs no reference rows
    # group 2: no queries vs r8..r9
    # group 3: q6..q9 vs r10..r15 with r11 all NaN and r12 a rolled copy of q7
    r[11] = np.nan
    r[12] = rolled(q[7], 0)
    # group 4: q10..q13 vs r16..r23 where r17 == r20 and both are the closest row to q10 at shift 3
    r[17] = rolled(q[10], 3) + np.float32(0.001)
    r[20] = r[17]
    qo = np.array([0, 4, 6, 6, 10, 14], np.int64)
    ro = np.array([0, 8, 8, 10, 16, 24], np.int64)
    return q, r, qo, ro


def check_against_numpy(q, r, qo, ro, best, shift, d, sd, rtol=1e-5):
    """The matcher's results against numpy's 12-shift minimum: distances within rtol, best/shift equal except where
    numpy's two best candidates are within rtol of each other.  -> number of queries checked."""
    n = 0
    for g in range(len(qo) - 1):
        qs, rs = slice(qo[g], qo[g + 1]), slice(ro[g], ro[g + 1])
        if qo[g + 1] == qo[g]:
            continue
        D = numpy_shift_distances(q[qs], r[rs]) if ro[g + 1] > ro[g] else np.zeros((qo[g + 1] - qo[g], 0, L))
        for i in range(qo[g + 1] - qo[g]):
            o = qo[g] + i - qo[0]
            Di = D[i]
            fin = np.isfinite(Di)
            if not fin.any():
                assert best[o] == -1 and shift[o] == -1 and np.isposinf(d[o]) and np.isposinf(sd[o])
                n += 1
                continue
            flat = np.where(fin, Di, np.inf).reshape(-1)
            k = int(np.argmin(flat))
            row_min = np.where(fin, Di, np.inf).min(axis=1)
            exp_d = flat[k]
            assert abs(float(d[o]) - exp_d) <= rtol * max(exp_d, 1e-30) + 1e-30, (g, i, d[o], exp_d)
            others = np.delete(row_min, k // L)
            exp_sd = others.min() if len(others) else np.inf
            if np.isfinite(exp_sd):
                assert abs(float(sd[o]) - exp_sd) <= rtol * max(exp_sd, 1e-30) + 1e-30, (g, i, sd[o], exp_sd)
            else:
                assert np.isposinf(sd[o])
            srt = np.sort(flat)
            if len(srt) < 2 or srt[1] - srt[0] > rtol * max(srt[1], 1e-30):
                assert best[o] == ro[g] + k // L and shift[o] == k % L, (g, i, best[o], shift[o], k)
            n += 1
    return n
