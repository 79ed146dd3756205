"""The CPU restatement of fe_match_descriptors (match_oracle/fe_match_oracle.cpp): against an independent float64
evaluation of the 12-shift minimum, and the exact properties the contract in include/fe_b200.h promises."""
import numpy as np

from match_oracle import binding as mo
from match_cases import (check_against_numpy, constructed, random_rows, rolled, to_records)


def test_oracle_agrees_with_numpy_on_random_rows():
    rng = np.random.default_rng(11)
    q = random_rows(rng, 20)
    r = random_rows(rng, 45)
    qo = np.array([0, 7, 7, 20], np.int64)
    ro = np.array([0, 30, 33, 45], np.int64)
    res = mo.match_descriptors(q, r, qo, ro, n_threads=4)
    assert check_against_numpy(q, r, qo, ro, *res) == 20


def test_oracle_agrees_with_numpy_on_real_descriptors(ob, synth):
    P = ob.node_default()
    pts, offs, rp = synth.generate(2, 12)
    ko, kp, d, _ = ob.process_batch(P, pts, offs, rp, mode=1, n_threads=4)
    assert len(d) > 10
    # scan s against scan s - 1, then everything against everything
    qo, ro = ko[1:], ko[:-1]
    res = mo.match_descriptors(d, d, qo, ro, n_threads=4)
    assert check_against_numpy(d, d, qo, ro, *res) == ko[-1] - ko[1]
    best, shift, dist2, sd = mo.match_descriptors(d, d, n_threads=4)
    assert check_against_numpy(d, d, np.array([0, len(d)]), np.array([0, len(d)]), best, shift, dist2, sd) == len(d)
    # every finite row finds itself at shift 0
    fin = np.isfinite(d).all(axis=1)
    assert np.array_equal(best[fin], np.nonzero(fin)[0]) and (shift[fin] == 0).all() and (dist2[fin] == 0).all()
    assert (best[~fin] == -1).all()


def test_oracle_exact_properties():
    rng = np.random.default_rng(5)
    q, r, qo, ro = constructed(rng)
    best, shift, d, sd = mo.match_descriptors(q, r, qo, ro)
    assert len(best) == 14
    # rolled copy: distance exactly 0 at the right shift
    assert best[1] == 3 and shift[1] == 5 and d[1] == 0.0
    # duplicated reference row: the lower index wins, second == best
    assert best[2] == 6 and shift[2] == 11 and d[2] == 0.0 and sd[2] == 0.0
    # NaN query row, and queries of a group without reference rows
    for i in (3, 4, 5):
        assert best[i] == -1 and shift[i] == -1 and np.isposinf(d[i]) and np.isposinf(sd[i])
    # a NaN reference row never matches; r12 is q7 itself
    assert best[7] == 12 and shift[7] == 0 and d[7] == 0.0
    assert (best[6:10] != 11).all()
    # a tie between two distinct rows at a non-zero distance
    assert best[10] == 17 and shift[10] == 3 and d[10] > 0 and sd[10] == d[10]
    assert check_against_numpy(q, r, qo, ro, best, shift, d, sd) == 14


def test_oracle_groups_edge_cases():
    rng = np.random.default_rng(6)
    q = random_rows(rng, 9)
    r = random_rows(rng, 12)
    r[10] = rolled(q[8], 7)
    # G = 0: nothing
    res = mo.match_descriptors(q, r, [3], [5])
    assert all(len(a) == 0 for a in res)
    # qo[0] > 0 and ro[0] > 0: output row i is query row qo[0] + i, best is an absolute row index
    best, shift, d, sd = mo.match_descriptors(q, r, [6, 8, 9], [2, 6, 12])
    assert len(best) == 3 and best[2] == 10 and shift[2] == 7 and d[2] == 0.0
    assert all(2 <= b < 6 for b in best[:2])
    full = mo.match_descriptors(q, r, [0, 6, 8, 9], [0, 2, 6, 12])
    for a, b in zip(full, (best, shift, d, sd)):
        assert np.array_equal(np.asarray(a)[6:].view(np.uint8), np.asarray(b).view(np.uint8))


def test_oracle_records_equal_bins():
    rng = np.random.default_rng(7)
    q, r, qo, ro = constructed(rng)
    a = mo.match_descriptors(q, r, qo, ro)
    b = mo.match_descriptors(to_records(q), to_records(r), qo, ro)
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))
