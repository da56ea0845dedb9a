"""GPU tests of sw_align_db / Engine.align_db: the CIGAR of the located best alignment of selected pairs of the
resident database.  The checks use strings and the scalar oracle's score only, so no traceback code is shared
between the kernel and the check: the ops consume exactly the located stretches, '=' / 'X' runs hold equal / unequal
bases, runs are maximal, both ends are '=', and the ops score S under the combined-gap rule.  A small pure-Python
rectangle DP with the header's tie rules reproduces the exact ops on seeded samples."""
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.test_gpu_locate import _all_pairs, _check_located, _code, _planted, _revcomp, _state
from tests.test_gpu_parity import _oracle_matrix, _rand
from tests.test_gpu_round2 import _overflow_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = "MIDNSHP=X"
DEFAULT = (5, -4, -12, -4)


def _runs(ops):
    return [(int(o) >> 4, OPS[int(o) & 15]) for o in ops]


def _op_score(runs, params, one_gap=True):
    """Score of the ops: a maximal run of I / D columns in any mix costs go + ge * length (one_gap=False prices each
    I or D run as a gap of its own)."""
    match, mismatch, go, ge = params
    total, gap = 0, 0
    for ln, op in runs + [(0, "=")]:
        if op in "ID":
            if gap and not one_gap and op != prev:
                total += go + ge * gap
                gap = 0
            gap += ln
        else:
            if gap:
                total += go + ge * gap
                gap = 0
            total += ln * (match if op == "=" else mismatch)
        prev = op
    return total


def _ref_ops(q, s, c, params):
    """The header's definition: rectangle DP with the h / u / g tie rules, then the walk from the end in state M."""
    match, mismatch, go, ge = params
    goe = go + ge
    qb, qe, sb, se = (int(x) for x in c)
    a, b = q[qb:qe], s[sb:se]
    m, n = len(a), len(b)
    gb = max(goe, ge)
    H = [[0] * (n + 1) for _ in range(m + 1)]
    G = [[gb] * (n + 1) for _ in range(m + 1)]
    d = [[0] * (n + 1) for _ in range(m + 1)]
    for i in range(1, m + 1):
        Hi, Hp, Gi, Gp, di = H[i], H[i - 1], G[i], G[i - 1], d[i]
        ai = a[i - 1]
        for j in range(1, n + 1):
            M = max(0, Hp[j - 1] + (match if ai == b[j - 1] else mismatch))
            up, left = Gp[j], Gi[j - 1]
            I = max(up, left)
            Gi[j] = max(M + goe, I + ge)
            Hi[j] = max(M, I)
            di[j] = (M < I) | (up < left) << 1 | (M + goe < I + ge) << 2
    cols = []
    i, j, st = m, n, "M"
    while True:
        assert i >= 1 and j >= 1, "the walk left the rectangle"
        if st == "M":
            cols.append("=" if a[i - 1] == b[j - 1] else "X")
            if (i, j) == (1, 1):
                break
            i, j = i - 1, j - 1
            assert i >= 1 and j >= 1, "the walk left the rectangle"
            st = "I" if d[i][j] & 1 else "M"
        else:
            if d[i][j] & 2:
                cols.append("D")
                j -= 1
            else:
                cols.append("I")
                i -= 1
            assert i >= 1 and j >= 1, "the walk left the rectangle"
            st = "I" if d[i][j] & 4 else "M"
    cols.reverse()
    runs = []
    for op in cols:
        if runs and runs[-1][1] == op:
            runs[-1][0] += 1
        else:
            runs.append([1, op])
    return [(ln, op) for ln, op in runs]


def _check_aligned(q, s, S, c, ops, params, msg=""):
    """The ops of one pair against its strings and located result."""
    runs = _runs(ops)
    if S == 0:
        assert runs == [], msg
        return runs
    qb, qe, sb, se = (int(x) for x in c)
    qi, si = qb, sb
    for k, (ln, op) in enumerate(runs):
        assert ln >= 1 and op in "=XID", (runs, msg)
        if k:
            assert op != runs[k - 1][1], ("runs not maximal", runs, msg)
        if op in "=X":
            for t in range(ln):
                assert (q[qi + t] == s[si + t]) == (op == "="), (runs, msg)
            qi += ln
            si += ln
        elif op == "I":
            qi += ln
        else:
            si += ln
    assert (qi, si) == (qe, se), ("ops do not consume the located stretches", runs, c, msg)
    assert runs[0][1] == "=" and runs[-1][1] == "=", (runs, msg)
    assert _op_score(runs, params) == S, (runs, S, msg)
    assert len(runs) <= (qe - qb) + (se - sb) - 1, msg
    return runs


def _pair_ops(cigar_off, cigar, k):
    return cigar[int(cigar_off[k]):int(cigar_off[k + 1])]


def _align_checked(e, rows, idx, seqs, subjects, params=DEFAULT, ref_sample=0, seed=0):
    """align_db of the pairs: score and coord equal locate_db's, every pair passes the full check, and a seeded
    sample of ref_sample pairs (all if ref_sample < 0) has exactly the reference's ops."""
    rows = np.asarray(rows, np.uint32)
    idx = np.asarray(idx, np.uint64)
    sc, co, off, cig = e.align_db(rows, idx)
    lsc, lco = e.locate_db(rows, idx)
    assert sc.dtype == np.int32 and co.dtype == np.uint32 and off.dtype == np.uint64 and cig.dtype == np.uint32
    assert co.shape == (len(rows), 4) and off.shape == (len(rows) + 1,) and off[0] == 0 and off[-1] == len(cig)
    np.testing.assert_array_equal(sc, lsc)
    np.testing.assert_array_equal(co, lco)
    for k in range(len(rows)):
        _check_aligned(seqs[rows[k]], subjects[idx[k]], int(sc[k]), co[k], _pair_ops(off, cig, k), params,
                       f"row {rows[k]} subject {idx[k]}")
    pick = range(len(rows)) if ref_sample < 0 else random.Random(seed).sample(range(len(rows)), min(ref_sample, len(rows)))
    for k in pick:
        if sc[k] > 0:
            want = _ref_ops(seqs[rows[k]], subjects[idx[k]], co[k], params)
            assert _runs(_pair_ops(off, cig, k)) == want, (k, want)
    return sc, co, off, cig


def _engine_db(pkg, queries, subjects, strands=False, **kw):
    e = pkg.Engine(**kw)
    if strands:
        e.set_strands(True)
    e.set_queries(queries)
    e.load_db(subjects)
    e.score_db()
    e.wait()
    return e


def test_align_query_lengths(oracle_mod, pkg):
    """Queries across the 16-row strip boundaries against ragged subjects with interior alignments."""
    rng = random.Random(71)
    queries = [_rand(rng, n) for n in (1, 15, 16, 17, 33, 150, 300)]
    subjects = _planted(rng, queries, 90)
    with _engine_db(pkg, queries, subjects) as e:
        rows, idx = _all_pairs(len(queries), len(subjects))
        sc, co, off, cig = _align_checked(e, rows, idx, queries, subjects, ref_sample=150, seed=71)
        assert e.device_error_bits == 0
    runs = [_runs(_pair_ops(off, cig, k)) for k in range(len(sc))]
    assert sum(any(op in "ID" for _, op in r) for r in runs) > 50      # indels inside many alignments
    assert sum(any(op == "X" for _, op in r) for r in runs) > 50
    o = oracle_mod.Oracle()
    for k in range(0, len(sc), 9):                                      # locate's definition still holds
        _check_located(o, queries[rows[k]], subjects[idx[k]], int(sc[k]), co[k])


def test_align_homopolymer_indels_and_ties(pkg):
    """A one-base indel in a homopolymer run lands on the run's first base; tandem repeats and duplicated queries."""
    rng = random.Random(72)
    left = _rand(rng, 39) + "C"
    right = "G" + _rand(rng, 39)
    ins_q, ins_s = left + "A" * 9 + right, left + "A" * 8 + right      # the query has one A more: an I
    del_q, del_s = left + "T" * 7 + right, left + "T" * 8 + right      # the subject has one T more: a D
    core = _rand(rng, 60)
    ac = "AC" * 20
    queries = [ins_q, del_q, core, ac, ac + _rand(rng, 30), "CA" * 13 + "C", core]
    subjects = [ins_s, del_s,
                "T" * 17 + core + _rand(rng, 20) + core + "T" * 17,
                "T" * 17 + "AC" * 30 + "T" * 17,
                _rand(rng, 40) + "AC" * 35 + _rand(rng, 40),
                "ACA" + "CA" * 12 + "GGG" + "AC" * 15,
                core + core,
                _rand(rng, 100) + ac[:25] + _rand(rng, 9) + ac[:25]]
    with _engine_db(pkg, queries, subjects) as e:
        rows, idx = _all_pairs(len(queries), len(subjects))
        sc, co, off, cig = _align_checked(e, rows, idx, queries, subjects, ref_sample=-1)
        assert e.device_error_bits == 0
    ns = len(subjects)
    got = {(int(rows[k]), int(idx[k])): pkg.cigar_str(_pair_ops(off, cig, k)) for k in range(len(sc))}
    assert got[0, 0] == "40=1I48="
    assert got[1, 1] == "40=1D47="
    assert got[2, 2] == "60=" and tuple(co[2 * ns + 2]) == (0, 60, 17, 77)
    for s in range(ns):
        assert got[2, s] == got[6, s]                                  # duplicated query: identical ops


def test_align_score_zero_and_empty(pkg):
    """Score 0 and empty subjects give no ops; n = 0 gives cigar_off = [0]."""
    queries = ["A" * 20, "ACGTACGT", "G"]
    subjects = ["", "C" * 30, "ACGTTT", "", "T", "GGGG"]
    with _engine_db(pkg, queries, subjects) as e:
        rows, idx = _all_pairs(len(queries), len(subjects))
        sc, co, off, cig = _align_checked(e, rows, idx, queries, subjects, ref_sample=-1)
        assert (sc == 0).sum() >= 8
        assert all(off[k] == off[k + 1] for k in range(len(sc)) if sc[k] == 0)
        sc0, co0, off0, cig0 = e.align_db([], [])
        assert sc0.shape == (0,) and co0.shape == (0, 4) and off0.tolist() == [0] and cig0.size == 0
    with _engine_db(pkg, queries, ["", ""]) as e:
        sc, co, off, cig = e.align_db([0, 1, 2], [1, 0, 1])
        assert (sc == 0).all() and (co == 0).all() and off.tolist() == [0, 0, 0, 0] and cig.size == 0


def test_align_both_strands(pkg):
    """Row nq + i is aligned as the reverse complement of query i; a palindrome's two rows give identical ops."""
    rng = random.Random(73)
    half = _rand(rng, 22)
    pal = half + _revcomp(half)
    queries = [_rand(rng, 120), pal, _rand(rng, 45)]
    rowseq = queries + [_revcomp(q) for q in queries]
    subjects = _planted(rng, rowseq, 60)
    with _engine_db(pkg, queries, subjects, strands=True) as e:
        assert e.nq == 6
        rows, idx = _all_pairs(6, len(subjects))
        sc, co, off, cig = _align_checked(e, rows, idx, rowseq, subjects, ref_sample=60, seed=73)
        assert e.device_error_bits == 0
    ns = len(subjects)
    for s in range(ns):
        assert _pair_ops(off, cig, ns + s).tolist() == _pair_ops(off, cig, 4 * ns + s).tolist()
    assert (sc[3 * ns:] > 0).sum() > 20


@pytest.mark.parametrize("params", [(5, -4, -8, -4), (5, -4, -2, -1), (5, -4, 4, -4)])
def test_align_parameter_sets(pkg, params):
    """Non-default penalties.  With 5/-4/-2/-1 a two-base substitution is cheaper as I and D columns priced as one
    gap (go + 4 ge = -6) than as two mismatches (-8), so some CIGAR has an I run next to a D run that scores S only
    under the combined-gap rule."""
    rng = random.Random(74)
    kw = dict(zip(("match", "mismatch", "gap_open", "gap_extend"), params))
    queries = [_rand(rng, n) for n in (17, 90, 150)]
    subjects = _planted(rng, queries, 50)
    flank_l, flank_r = _rand(rng, 30), _rand(rng, 30)
    queries.append(flank_l + "AC" + flank_r)
    subjects.append(flank_l + "GT" + flank_r)
    with _engine_db(pkg, queries, subjects, **kw) as e:
        rows, idx = _all_pairs(len(queries), len(subjects))
        sc, co, off, cig = _align_checked(e, rows, idx, queries, subjects, params=params, ref_sample=80, seed=74)
        assert e.device_error_bits == 0
    if params == (5, -4, -2, -1):
        mixed = 0
        for k in range(len(sc)):
            runs = _runs(_pair_ops(off, cig, k))
            if any(a[1] in "ID" and b[1] in "ID" for a, b in zip(runs, runs[1:])):
                assert _op_score(runs, params) == sc[k]
                mixed += _op_score(runs, params, one_gap=False) != sc[k]
        assert mixed >= 1


def test_align_score_beyond_16_bits(pkg):
    """A 6 700-nt identical pair scoring 33 500 gives 6700=."""
    rng = random.Random(75)
    s, subjects = _overflow_case(rng)
    queries = [s, _rand(rng, 150)]
    with _engine_db(pkg, queries, subjects) as e:
        sc, co, off, cig = _align_checked(e, [0, 0, 0, 1], [0, 3, 4, 7], queries, subjects)
        assert e.device_error_bits == 0
    assert sc[0] == 33500 and tuple(co[0]) == (0, 6700, 0, 6700)
    assert pkg.cigar_str(_pair_ops(off, cig, 0)) == "6700="


def test_align_shards(pkg):
    """Pairs spanning the shards in shuffled order with duplicates: identical to a one-GPU handle."""
    rng = random.Random(76)
    queries = [_rand(rng, n) for n in (150, 31, 260)]
    subjects = _planted(rng, queries, 3000)
    rows = np.array([rng.randrange(len(queries)) for _ in range(5000)], np.uint32)
    idx = np.array([rng.randrange(len(subjects)) for _ in range(5000)], np.uint64)
    rows = np.concatenate([rows, rows[:700]])
    idx = np.concatenate([idx, idx[:700]])
    perm = np.random.default_rng(76).permutation(len(rows))
    rows, idx = rows[perm], idx[perm]
    with _engine_db(pkg, queries, subjects) as e:
        want = _align_checked(e, rows, idx, queries, subjects, ref_sample=50, seed=76)
    for gpu_ids in ([0, 0, 0], list(range(pkg.device_count())) + [0]):
        with _engine_db(pkg, queries, subjects, gpu_ids=gpu_ids) as e:
            got = e.align_db(rows, idx)
            assert e.device_error_bits == 0
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b, err_msg=str(gpu_ids))


def test_align_with_hits_and_subject_best(pkg):
    """An align call between score_db and the fetch changes neither the fetched result nor the last call's cells,
    kernel name and kernel time; aligning the fetched pairs gives their scores."""
    rng = random.Random(77)
    queries = [_rand(rng, n) for n in (150, 70, 151)]
    subjects = _planted(rng, queries, 4000)
    ns = len(subjects)
    some_rows = np.array([rng.randrange(len(queries)) for _ in range(300)], np.uint32)
    some_idx = np.array([rng.randrange(ns) for _ in range(300)], np.uint64)
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.set_hits(60)
        e.score_db()
        ref = e.fetch_db_hits()
        e.score_db()
        e.align_db(some_rows, some_idx)                         # queued behind the unfetched scoring
        for a, b in zip(e.fetch_db_hits(), ref):
            np.testing.assert_array_equal(a, b)
        e.score_db()
        e.wait()
        before = _state(e)
        sc, co, off, cig = e.align_db(ref[0], ref[1])
        assert _state(e) == before
        for a, b in zip(e.fetch_db_hits(), ref):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(sc, ref[2])
        assert len(ref[0]) > 500
        for k in range(0, len(sc), 20):
            _check_aligned(queries[ref[0][k]], subjects[ref[1][k]], int(sc[k]), co[k], _pair_ops(off, cig, k), DEFAULT)

        e.set_hits(0)
        e.set_subject_best(True)
        e.score_db()
        ref = e.fetch_db_subject_best()
        e.score_db()
        e.align_db(some_rows, some_idx)
        for a, b in zip(e.fetch_db_subject_best(), ref):
            np.testing.assert_array_equal(a, b)
        e.score_db()
        e.wait()
        before = _state(e)
        sc, co, off, cig = e.align_db(ref[1], np.arange(ns))
        assert _state(e) == before
        for a, b in zip(e.fetch_db_subject_best(), ref):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(sc, ref[0])
        for k in range(0, ns, 20):
            _check_aligned(queries[ref[1][k]], subjects[k], int(sc[k]), co[k], _pair_ops(off, cig, k), DEFAULT)
        assert e.device_error_bits == 0


def _raw_align(lib, e, rows, idx, cap, with_cigar=True):
    """sw_align_db through ctypes with sentinel-filled outputs: (rc, count, score, coord, cigar_off, cigar)."""
    import ctypes as C
    n = len(rows)
    rows = np.asarray(rows, np.uint32)
    idx = np.asarray(idx, np.uint64)
    score = np.full(n, -7, np.int32)
    coord = np.full((n, 4), 7, np.uint32)
    off = np.full(n + 1, 7, np.uint64)
    cig = np.full(max(cap, 1), 7, np.uint32)
    count = C.c_size_t(12345)
    rc = lib.sw_align_db(e.h, rows.ctypes.data, idx.ctypes.data, n, score.ctypes.data, coord.ctypes.data,
                         off.ctypes.data, cig.ctypes.data if with_cigar else None, cap, C.byref(count))
    return rc, count.value, score, coord, off, cig


def test_align_contract(pkg, monkeypatch):
    lib = pkg.load_library()
    rng = random.Random(78)
    queries = [_rand(rng, 150), _rand(rng, 80)]
    subjects = _planted(rng, queries, 500)
    ns = len(subjects)
    rows = np.array([rng.randrange(2) for _ in range(400)], np.uint32)
    idx = np.array([rng.randrange(ns) for _ in range(400)], np.uint64)
    with pkg.Engine() as e:
        e.set_queries(queries)
        assert _code(pkg, lambda: e.align_db([0], [0])) == pkg.SW_ESTATE         # no database
        e.load_db(subjects)
        e.score_db()
        launches = e.kernel_launches
        assert _code(pkg, lambda: e.align_db([2], [0])) == pkg.SW_EINVAL        # row out of range
        assert _code(pkg, lambda: e.align_db([0, 1], [0, ns])) == pkg.SW_EINVAL  # index out of range
        r, i = np.zeros(1, np.uint32), np.zeros(1, np.uint64)
        sc, co = np.zeros(1, np.int32), np.zeros(4, np.uint32)
        off, cig = np.zeros(2, np.uint64), np.zeros(400, np.uint32)
        import ctypes as C
        cnt = C.c_size_t(0)
        args = [r.ctypes.data, i.ctypes.data, 1, sc.ctypes.data, co.ctypes.data, off.ctypes.data, cig.ctypes.data, 400,
                C.byref(cnt)]
        for k in (0, 1, 3, 4, 5, 8):                            # row, index, score, coord, cigar_off, count
            a = list(args)
            a[k] = None
            assert lib.sw_align_db(e.h, *a) == pkg.SW_EINVAL, k
        a = list(args)
        a[6] = None                                              # cigar NULL with cap > 0
        assert lib.sw_align_db(e.h, *a) == pkg.SW_EINVAL
        assert lib.sw_align_db(e.h, None, None, 0, None, None, None, None, 0, None) == pkg.SW_OK
        assert lib.sw_align_db(e.h, None, None, 0, None, None, off.ctypes.data, None, 0, C.byref(cnt)) == pkg.SW_OK
        assert off[0] == 0 and cnt.value == 0
        assert e.kernel_launches == launches
        good = _align_checked(e, rows, idx, queries, subjects)
        assert e.kernel_launches > launches
        total = len(good[3])
        assert total > 400
        # the size query, then too small a buffer: the exact count and nothing else written; a retry recomputes
        rc, count, *_ = _raw_align(lib, e, rows, idx, 0, with_cigar=False)
        assert rc == pkg.SW_ECAPACITY and count == total
        rc, count, score, coord, off2, cig2 = _raw_align(lib, e, rows, idx, total - 1)
        assert rc == pkg.SW_ECAPACITY and count == total
        assert (score == -7).all() and (coord == 7).all() and (off2 == 7).all() and (cig2 == 7).all()
        rc, count, score, coord, off2, cig2 = _raw_align(lib, e, rows, idx, total)
        assert rc == pkg.SW_OK and count == total
        for a, b in zip((score, coord, off2, cig2), good):
            np.testing.assert_array_equal(a, b)
        # a batch in flight: SW_EAGAIN; sw_score_batch reused the database's buffers: SW_ESTATE
        e.set_small_batch_path(False)
        e.score_batch(subjects[:300])
        assert _code(pkg, lambda: e.align_db([0], [0])) == pkg.SW_EAGAIN
        e.fetch()
        assert _code(pkg, lambda: e.align_db([0], [0])) == pkg.SW_ESTATE
        e.load_db(subjects)
        for a, b in zip(e.align_db(rows, idx), good):
            np.testing.assert_array_equal(a, b)
        assert e.device_error_bits == 0
    # a budget of a few pairs' rectangles: many rounds, the same result
    monkeypatch.setenv("SW_B200_ALIGN_SCRATCH_MB", "0.05")
    with _engine_db(pkg, queries, subjects) as e:
        launches = e.kernel_launches
        got = e.align_db(rows, idx)
        assert e.kernel_launches - launches >= 1 + 5                # the locate launch, then the rounds
        assert e.device_error_bits == 0
    for a, b in zip(got, good):
        np.testing.assert_array_equal(a, b)
    # a budget below one pair's rectangle: SW_ERANGE, nothing written
    monkeypatch.setenv("SW_B200_ALIGN_SCRATCH_MB", "0.001")
    with _engine_db(pkg, queries, subjects) as e:
        rc, count, score, coord, off2, cig2 = _raw_align(lib, e, rows, idx, total)
        assert rc == pkg.SW_ERANGE
        assert count == 12345 and (score == -7).all() and (coord == 7).all() and (off2 == 7).all() and (cig2 == 7).all()
        assert e.device_error_bits == 0
    monkeypatch.delenv("SW_B200_ALIGN_SCRATCH_MB")
    with pkg.Engine(score_width=12) as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        launches = e.kernel_launches
        assert _code(pkg, lambda: e.align_db([0], [0])) == pkg.SW_EINVAL       # the wrapping machine
        assert e.kernel_launches == launches


def test_align_large_job(pkg):
    """1.2 M x 150 nt with planted homologs against 100 queries in hits mode at T = 200: every hit aligned with its
    ops scoring the hit's score, 2 000 sampled hits given the full check (200 of them against the reference)."""
    q = pkg.random_packed_db(100, 150, seed=94)
    db = pkg.random_packed_db(1_200_000, 150, seed=95)
    pkg.plant_homologs(db, q, 0.01, seed=96)
    with pkg.Engine() as e:
        e.set_queries(q)
        e.load_db(db)
        e.set_hits(200)
        e.score_db()
        row, idx, hsc = e.fetch_db_hits()
        sc, co, off, cig = e.align_db(row, idx)
        lsc, lco = e.locate_db(row, idx)
        assert e.device_error_bits == 0
    assert 5_000 < len(row) < 1_000_000
    np.testing.assert_array_equal(sc, hsc)
    np.testing.assert_array_equal(sc, lsc)
    np.testing.assert_array_equal(co, lco)
    for k in range(len(row)):
        assert _op_score(_runs(_pair_ops(off, cig, k)), DEFAULT) == sc[k], k
    sample = np.random.default_rng(97).choice(len(row), 2000, replace=False)
    for n, k in enumerate(sample):
        qs = pkg.seqio.unpack_to_str(q[0], int(q[1][row[k]]), int(q[2][row[k]]))
        ss = pkg.seqio.unpack_to_str(db[0], int(db[1][idx[k]]), int(db[2][idx[k]]))
        _check_aligned(qs, ss, int(sc[k]), co[k], _pair_ops(off, cig, k), DEFAULT, f"hit {k}")
        if n < 200:
            assert _runs(_pair_ops(off, cig, k)) == _ref_ops(qs, ss, co[k], DEFAULT), k


def test_align_golden_and_cli(golden, pkg, tmp_path):
    """query100.fa x data500.fa through the CLI: -T ... -A and -B -A append the span and a CIGAR that pass the full
    check; -A alone is a usage error; without -A the lines are unchanged."""
    q = golden["fasta"]["query100.fa"][0][1]
    db = golden["fasta"]["data500.fa"]
    seq = dict(db)
    cli = os.path.join(ROOT, "bin", "sw_b200_cli")
    qf, lf = tmp_path / "query100.fa", tmp_path / "data500.fa"
    qf.write_text(">query\n" + q + "\n")
    lf.write_text("".join(f">{n}\n{s}\n" for n, s in db))
    tail = r" query (\d+)-(\d+) subject (\d+)-(\d+) cigar (\*|(?:\d+[=XID])+)$"

    def check(name, score, m):
        qb, qe, sb, se = (int(x) for x in m.groups()[:4])
        text = m.group(5)
        ops = [] if text == "*" else [int(n) << 4 | OPS.index(op) for n, op in re.findall(r"(\d+)([=XID])", text)]
        if score == 0:
            assert (qb, qe, sb, se) == (0, 0, 0, 0) and text == "*"
        else:
            _check_aligned(q, seq[name], score, (qb - 1, qe, sb - 1, se), ops, DEFAULT, name)
            assert [(ln, op) for ln, op in _runs(ops)] == _ref_ops(q, seq[name], (qb - 1, qe, sb - 1, se), DEFAULT)

    base = [os.path.abspath(cli), "-q", str(qf), "-l", str(lf), "-t", "30"]
    for mode, pat in ((["-T", "40"], r"(\S+) x (\S+) result: (-?\d+), biased: -?\d+\(0x[0-9a-f]+\)"),
                      (["-B"], r"(\S+) best (\S+) result: (-?\d+), second: (-?\d+)")):
        plain = subprocess.run(base + mode, capture_output=True, text=True, timeout=120)
        located = subprocess.run(base + mode + ["-L"], capture_output=True, text=True, timeout=120)
        r = subprocess.run(base + mode + ["-A"], capture_output=True, text=True, timeout=120)
        assert plain.returncode == 0 and located.returncode == 0 and r.returncode == 0, r.stdout + r.stderr
        lines = r.stdout.splitlines()
        assert len(lines) == len(plain.stdout.splitlines()) == len(located.stdout.splitlines()) > 10
        for line, pl, lo in zip(lines, plain.stdout.splitlines(), located.stdout.splitlines()):
            m = re.match(pat + tail, line)
            assert m and line.startswith(lo + " cigar ") and lo.startswith(pl + " query "), line
            name = m.group(2) if mode[0] == "-T" else m.group(1)
            check(name, int(m.group(3)), re.search(tail, line))
    r = subprocess.run(base + ["-A"], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "-A" in r.stdout


def test_align_on_the_bounds_check_build(pkg):
    """This file again on libsw_b200_check.so (index checks on the direction buffer and op slots, the walk staying in
    the rectangle, ending at (1, 1) in M and scoring S, canaries)."""
    lib = os.path.join(ROOT, "smith-waterman-fpga-module_b200", "libsw_b200_check.so")
    if not os.path.exists(lib):
        pytest.skip("libsw_b200_check.so not built (make -C csrc CHECK=1)")
    if pkg.is_check_build():
        pytest.skip("already running the check build")
    env = dict(os.environ, SW_B200_LIB=lib)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu",
                        "-k", "not bounds_check_build", "-p", "no:cacheprovider"], capture_output=True, text=True, env=env,
                       timeout=2400, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout
