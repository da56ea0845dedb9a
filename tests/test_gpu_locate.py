"""GPU tests of sw_locate_db / Engine.locate_db: begin and end of the best local alignment of selected pairs of the
resident database.  The definition (include/sw_b200.h) is pinned with the scalar oracle's score on strings only, so
no coordinate code is shared between the kernel and the check: for S > 0 the end is the first column (then row)
where a prefix reaches S, and the begin is the last column (then row) from which the stretch up to the end still
reaches S.  Together with the matched end bases these conditions fix the 5-tuple uniquely."""
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.test_gpu_parity import _mutate, _oracle_matrix, _rand
from tests.test_gpu_round2 import _overflow_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def _revcomp(s):
    return "".join(COMP[c] for c in reversed(s))


def _check_located(o, q, s, S, c, msg=""):
    qb, qe, sb, se = (int(x) for x in c)
    if S == 0:
        assert (qb, qe, sb, se) == (0, 0, 0, 0), msg
        return
    assert 0 <= qb < qe <= len(q) and 0 <= sb < se <= len(s), (c, msg)
    # the end: the first column, then the first row, where the prefixes reach S
    assert o.score(q[:qe], s[:se]) == S, msg
    assert o.score(q, s[:se - 1]) < S, msg
    assert o.score(q[:qe - 1], s[:se]) < S, msg
    # the begin: the last column, then the last row, from which the stretch up to the end reaches S
    assert o.score(q[qb:qe], s[sb:se]) == S, msg
    assert o.score(q[:qe], s[sb + 1:se]) < S, msg
    assert o.score(q[qb + 1:qe], s[sb:se]) < S, msg
    # every parameter set here has mismatch < 0: both ends are matched base pairs
    assert q[qb] == s[sb] and q[qe - 1] == s[se - 1], msg


def _planted(rng, queries, n):
    """0-600 nt subjects: mutated stretches of the queries inside random flanks, some empty, some random."""
    subjects = []
    for _ in range(n):
        r = rng.random()
        if r < 0.05:
            subjects.append("")
        elif r < 0.15:
            subjects.append(_rand(rng, rng.randint(1, 600)))
        else:
            q = rng.choice(queries)
            a = rng.randrange(len(q))
            b = rng.randint(a + 1, len(q))
            core = _mutate(rng, q[a:b], 0.08, 0.04)
            subjects.append((_rand(rng, rng.randint(0, 200)) + core + _rand(rng, rng.randint(0, 200)))[:600])
    return subjects


def _all_pairs(rows, ns):
    r, s = np.meshgrid(np.arange(rows, dtype=np.uint32), np.arange(ns, dtype=np.uint64), indexing="ij")
    return r.reshape(-1), s.reshape(-1)


def _locate_all(e, queries, subjects, mat, o, rowseq=None):
    """Locates every pair of the resident database; checks each one against the oracle and the matrix entry."""
    rows, idx = _all_pairs(mat.shape[0], len(subjects))
    sc, co = e.locate_db(rows, idx)
    assert sc.dtype == np.int32 and co.dtype == np.uint32 and co.shape == (len(rows), 4)
    np.testing.assert_array_equal(sc, mat[rows, idx.astype(np.int64)])
    seqs = rowseq if rowseq is not None else queries
    for k in range(len(rows)):
        _check_located(o, seqs[rows[k]], subjects[idx[k]], int(sc[k]), co[k], f"row {rows[k]} subject {idx[k]}")
    return sc, co


def test_locate_query_lengths_vs_oracle(oracle_mod, pkg):
    """Queries across the 16-row strip boundaries against ragged subjects with interior alignments."""
    rng = random.Random(61)
    queries = [_rand(rng, n) for n in (1, 15, 16, 17, 33, 150, 300)]
    subjects = _planted(rng, queries, 90)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        np.testing.assert_array_equal(mat, want)
        sc, co = _locate_all(e, queries, subjects, mat, oracle_mod.Oracle())
        assert e.device_error_bits == 0
    pos = sc > 0
    assert ((co[:, 0] > 0) & (co[:, 2] > 0) & pos).sum() > 100          # begins inside both sequences
    assert ((co[:, 1] < np.array([len(queries[r]) for r in _all_pairs(len(queries), len(subjects))[0]])) & pos).sum() > 100


def test_locate_ties(oracle_mod, pkg):
    """Two identical planted copies: the end is in the first one.  Tandem repeats have several equal-score begins
    and ends.  Duplicated queries give identical rows."""
    rng = random.Random(62)
    o = oracle_mod.Oracle()
    core = _rand(rng, 60)
    flank = "T" * 17
    ac = "AC" * 20
    queries = [core, ac, ac + _rand(rng, 30), "CA" * 13 + "C", core]
    subjects = [flank + core + _rand(rng, 20) + core + flank,
                flank + "AC" * 30 + flank,
                _rand(rng, 40) + "AC" * 35 + _rand(rng, 40),
                "ACA" + "CA" * 12 + "GGG" + "AC" * 15,
                core + core,
                _rand(rng, 100) + ac[:25] + _rand(rng, 9) + ac[:25]]
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        np.testing.assert_array_equal(mat, want)
        sc, co = _locate_all(e, queries, subjects, mat, o)
        assert e.device_error_bits == 0
    ns = len(subjects)
    got = {(k // ns, k % ns): (int(sc[k]), tuple(int(x) for x in co[k])) for k in range(len(sc))}
    assert got[0, 0] == (300, (0, 60, 17, 77))                 # the first copy
    assert got[0, 4] == (300, (0, 60, 0, 60))
    assert got[1, 1] == (200, (0, 40, 17, 57))                 # the first 40-base run of AC repeats
    for s in range(ns):
        assert got[0, s] == got[4, s]                          # duplicated query


def test_locate_score_zero_and_empty(oracle_mod, pkg):
    """Zero-length subjects, all-mismatch pairs and pairs scoring 0 give all zeros; n = 0 is fine."""
    queries = ["A" * 20, "ACGTACGT", "G"]
    subjects = ["", "C" * 30, "ACGTTT", "", "T", "GGGG"]
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        np.testing.assert_array_equal(mat, want)
        sc, co = _locate_all(e, queries, subjects, mat, oracle_mod.Oracle())
        assert (sc[mat.reshape(-1) == 0] == 0).all() and (co[mat.reshape(-1) == 0] == 0).all()
        assert (mat == 0).sum() >= 8
        sc0, co0 = e.locate_db([], [])
        assert sc0.shape == (0,) and co0.shape == (0, 4)
    with pkg.Engine() as e:                                     # a database of empty subjects only
        e.set_queries(queries)
        e.load_db(["", ""])
        e.score_db()
        sc, co = e.locate_db([0, 1, 2], [1, 0, 1])
        assert (sc == 0).all() and (co == 0).all()


def test_locate_both_strands(oracle_mod, pkg):
    """Row nq + i is the reverse complement of query i; its coordinates are positions in that string."""
    rng = random.Random(63)
    half = _rand(rng, 22)
    pal = half + _revcomp(half)
    queries = [_rand(rng, 120), pal, _rand(rng, 45)]
    subjects = _planted(rng, queries + [_revcomp(q) for q in queries], 60)
    rowseq = queries + [_revcomp(q) for q in queries]
    assert _revcomp(pal) == pal
    with pkg.Engine() as e:
        e.set_strands(True)
        e.set_queries(queries)
        assert e.nq == 6
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        np.testing.assert_array_equal(mat, _oracle_matrix(oracle_mod, pkg, rowseq, subjects))
        sc, co = _locate_all(e, queries, subjects, mat, oracle_mod.Oracle(), rowseq=rowseq)
        assert e.device_error_bits == 0
    ns = len(subjects)
    np.testing.assert_array_equal(sc[ns:2 * ns], sc[4 * ns:5 * ns])     # the palindrome's two rows
    np.testing.assert_array_equal(co[ns:2 * ns], co[4 * ns:5 * ns])


@pytest.mark.parametrize("params", [(5, -4, -8, -4), (5, -4, -2, -1), (5, -4, 4, -4)])
def test_locate_parameter_sets(oracle_mod, pkg, params):
    """Non-default penalties; with gap_open + gap_extend == 0 gap cells reach S too, which pins the M-based rule."""
    rng = random.Random(64)
    kw = dict(zip(("match", "mismatch", "gap_open", "gap_extend"), params))
    queries = [_rand(rng, n) for n in (17, 90, 150)]
    subjects = _planted(rng, queries, 50)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects, **kw)
    with pkg.Engine(**kw) as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        np.testing.assert_array_equal(mat, want)                # the scan itself first
        _locate_all(e, queries, subjects, mat, oracle_mod.Oracle(**kw))
        assert e.device_error_bits == 0


def test_locate_scores_beyond_16_bits(oracle_mod, pkg):
    """The located score is the exact int32 matrix entry above 32 767 too."""
    rng = random.Random(65)
    s, subjects = _overflow_case(rng)
    queries = [s, _rand(rng, 150)]
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        assert mat[0, 0] == 33500 and (mat > 32767).sum() >= 2
        sc, co = _locate_all(e, queries, subjects, mat, oracle_mod.Oracle())
        assert e.device_error_bits == 0
    assert sc[0] == 33500 and tuple(co[0]) == (0, 6700, 0, 6700)


def test_locate_shards(oracle_mod, pkg):
    """Pairs spanning the shards in shuffled order with duplicates: identical to a one-GPU handle."""
    rng = random.Random(66)
    queries = [_rand(rng, n) for n in (150, 31, 260)]
    subjects = _planted(rng, queries, 3000)
    nrows = len(queries)
    rows = np.array([rng.randrange(nrows) for _ in range(5000)], np.uint32)
    idx = np.array([rng.randrange(len(subjects)) for _ in range(5000)], np.uint64)
    rows = np.concatenate([rows, rows[:700]])
    idx = np.concatenate([idx, idx[:700]])
    perm = np.random.default_rng(66).permutation(len(rows))
    rows, idx = rows[perm], idx[perm]
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        want = e.locate_db(rows, idx)
    np.testing.assert_array_equal(want[0], mat[rows, idx.astype(np.int64)])
    o = oracle_mod.Oracle()
    for k in range(0, len(rows), 25):
        _check_located(o, queries[rows[k]], subjects[idx[k]], int(want[0][k]), want[1][k])
    for gpu_ids in ([0, 0, 0], list(range(pkg.device_count())) + [0]):
        with pkg.Engine(gpu_ids=gpu_ids) as e:
            e.set_queries(queries)
            e.load_db(subjects)
            e.score_db()
            got = e.locate_db(rows, idx)
            assert e.device_error_bits == 0
        np.testing.assert_array_equal(got[0], want[0], err_msg=str(gpu_ids))
        np.testing.assert_array_equal(got[1], want[1], err_msg=str(gpu_ids))


def _state(e):
    return e.last_cells, e.last_kernel_name, e.last_kernel_ms


def test_locate_with_hits_and_subject_best(oracle_mod, pkg):
    """A locate call between score_db and the fetch changes neither the fetched result nor the last call's
    cells, kernel name and kernel time; locating the fetched pairs gives their scores."""
    rng = random.Random(67)
    queries = [_rand(rng, n) for n in (150, 70, 151)]
    subjects = _planted(rng, queries, 4000)
    ns = len(subjects)
    some_rows = np.array([rng.randrange(len(queries)) for _ in range(300)], np.uint32)
    some_idx = np.array([rng.randrange(ns) for _ in range(300)], np.uint64)
    o = oracle_mod.Oracle()
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.set_hits(60)
        e.score_db()
        ref = e.fetch_db_hits()
        e.score_db()
        e.locate_db(some_rows, some_idx)                        # queued behind the unfetched scoring
        got = e.fetch_db_hits()
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a, b)
        e.score_db()
        e.wait()
        before = _state(e)
        sc, co = e.locate_db(ref[0], ref[1])
        assert _state(e) == before
        got = e.fetch_db_hits()
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(sc, ref[2])
        for k in range(0, len(sc), 20):
            _check_located(o, queries[ref[0][k]], subjects[ref[1][k]], int(sc[k]), co[k])
        assert len(ref[0]) > 500

        e.set_hits(0)
        e.set_subject_best(True)
        e.score_db()
        ref = e.fetch_db_subject_best()
        e.score_db()
        e.locate_db(some_rows, some_idx)
        got = e.fetch_db_subject_best()
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a, b)
        e.score_db()
        e.wait()
        before = _state(e)
        sc, co = e.locate_db(ref[1], np.arange(ns))
        assert _state(e) == before
        got = e.fetch_db_subject_best()
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(sc, ref[0])
        for k in range(0, ns, 20):
            _check_located(o, queries[ref[1][k]], subjects[k], int(sc[k]), co[k])
        assert e.device_error_bits == 0


def _code(pkg, fn):
    with pytest.raises(pkg.SwError) as ei:
        fn()
    return ei.value.code


def test_locate_contract(pkg):
    lib = pkg.load_library()
    rng = random.Random(68)
    queries = [_rand(rng, 150), _rand(rng, 80)]
    subjects = _planted(rng, queries, 500)
    ns = len(subjects)
    with pkg.Engine() as e:
        e.set_queries(queries)
        assert _code(pkg, lambda: e.locate_db([0], [0])) == pkg.SW_ESTATE         # no database
        e.load_db(subjects)
        e.score_db()
        launches = e.kernel_launches
        assert _code(pkg, lambda: e.locate_db([2], [0])) == pkg.SW_EINVAL        # row out of range
        assert _code(pkg, lambda: e.locate_db([0, 1], [0, ns])) == pkg.SW_EINVAL  # index out of range
        sc = np.zeros(1, np.int32)
        co = np.zeros(4, np.uint32)
        r = np.zeros(1, np.uint32)
        i = np.zeros(1, np.uint64)
        assert lib.sw_locate_db(e.h, None, i.ctypes.data, 1, sc.ctypes.data, co.ctypes.data) == pkg.SW_EINVAL
        assert lib.sw_locate_db(e.h, r.ctypes.data, None, 1, sc.ctypes.data, co.ctypes.data) == pkg.SW_EINVAL
        assert lib.sw_locate_db(e.h, r.ctypes.data, i.ctypes.data, 1, None, co.ctypes.data) == pkg.SW_EINVAL
        assert lib.sw_locate_db(e.h, r.ctypes.data, i.ctypes.data, 1, sc.ctypes.data, None) == pkg.SW_EINVAL
        assert lib.sw_locate_db(e.h, None, None, 0, None, None) == pkg.SW_OK
        assert e.kernel_launches == launches
        good = e.locate_db([1, 0], [ns - 1, 0])
        assert e.kernel_launches > launches
        # a batch in flight: SW_EAGAIN; sw_score_batch reused the database's buffers: SW_ESTATE
        for small in (True, False):
            e.set_small_batch_path(small)
            e.score_batch(subjects[:300])
            assert _code(pkg, lambda: e.locate_db([0], [0])) == pkg.SW_EAGAIN
            e.fetch()
            assert _code(pkg, lambda: e.locate_db([0], [0])) == pkg.SW_ESTATE
            e.load_db(subjects)
            again = e.locate_db([1, 0], [ns - 1, 0])
            for a, b in zip(again, good):
                np.testing.assert_array_equal(a, b)
        assert e.device_error_bits == 0
    with pkg.Engine(score_width=12) as e:
        e.set_queries(queries)
        e.load_db(subjects)
        e.score_db()
        launches = e.kernel_launches
        assert _code(pkg, lambda: e.locate_db([0], [0])) == pkg.SW_EINVAL       # the wrapping machine
        assert e.kernel_launches == launches


def test_locate_large_job(oracle_mod, pkg):
    """1.2 M x 150 nt with planted homologs against 100 queries in hits mode: every hit located, its score equal
    to the hit list's, a seeded sample of 2 000 checked against the oracle."""
    q = pkg.random_packed_db(100, 150, seed=94)
    db = pkg.random_packed_db(1_200_000, 150, seed=95)
    pkg.plant_homologs(db, q, 0.01, seed=96)
    with pkg.Engine() as e:
        e.set_queries(q)
        e.load_db(db)
        e.set_hits(200)
        e.score_db()
        row, idx, hsc = e.fetch_db_hits()
        sc, co = e.locate_db(row, idx)
        assert e.device_error_bits == 0
    assert 5_000 < len(row) < 1_000_000
    np.testing.assert_array_equal(sc, hsc)
    o = oracle_mod.Oracle()
    sample = np.random.default_rng(97).choice(len(row), 2000, replace=False)
    for k in sample:
        qs = pkg.seqio.unpack_to_str(q[0], int(q[1][row[k]]), int(q[2][row[k]]))
        ss = pkg.seqio.unpack_to_str(db[0], int(db[1][idx[k]]), int(db[2][idx[k]]))
        _check_located(o, qs, ss, int(sc[k]), co[k], f"hit {k}")


def test_locate_golden_and_cli(golden, oracle_mod, pkg, tmp_path):
    """query100.fa x data500.fa through the CLI: -T ... -L and -B -L append 1-based inclusive spans that satisfy
    the definition; -L alone is a usage error; without -L the lines are unchanged."""
    q = golden["fasta"]["query100.fa"][0][1]
    db = golden["fasta"]["data500.fa"]
    seq = dict(db)
    o = oracle_mod.Oracle()
    cli = os.path.join(ROOT, "bin", "sw_b200_cli")
    qf, lf = tmp_path / "query100.fa", tmp_path / "data500.fa"
    qf.write_text(">query\n" + q + "\n")
    lf.write_text("".join(f">{n}\n{s}\n" for n, s in db))
    span = r" query (\d+)-(\d+) subject (\d+)-(\d+)$"

    def check(name, score, m):
        qb, qe, sb, se = (int(x) for x in m.groups())
        if score == 0:
            assert (qb, qe, sb, se) == (0, 0, 0, 0)
        else:
            _check_located(o, q, seq[name], score, (qb - 1, qe, sb - 1, se), name)

    base = [os.path.abspath(cli), "-q", str(qf), "-l", str(lf), "-t", "30"]
    plain = subprocess.run(base + ["-T", "40"], capture_output=True, text=True, timeout=120)
    r = subprocess.run(base + ["-T", "40", "-L"], capture_output=True, text=True, timeout=120)
    assert plain.returncode == 0 and r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert len(lines) == len(plain.stdout.splitlines()) > 10
    for line, pl in zip(lines, plain.stdout.splitlines()):
        m = re.match(r"(\S+) x (\S+) result: (-?\d+), biased: -?\d+\(0x[0-9a-f]+\)" + span, line)
        assert m and line.startswith(pl + " query "), line
        check(m.group(2), int(m.group(3)), re.search(span, line))
    plain = subprocess.run(base + ["-B"], capture_output=True, text=True, timeout=120)
    r = subprocess.run(base + ["-B", "-L"], capture_output=True, text=True, timeout=120)
    assert plain.returncode == 0 and r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert len(lines) == len(db) == len(plain.stdout.splitlines())
    for line, pl in zip(lines, plain.stdout.splitlines()):
        m = re.match(r"(\S+) best (\S+) result: (-?\d+), second: (-?\d+)" + span, line)
        assert m and line.startswith(pl + " query "), line
        check(m.group(1), int(m.group(3)), re.search(span, line))
    r = subprocess.run(base + ["-L"], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "-L" in r.stdout


def test_locate_on_the_bounds_check_build(pkg):
    """This file again on libsw_b200_check.so (index checks on the query, subject and scratch reads and the result
    stores, the reverse pass reaching S, canaries)."""
    lib = os.path.join(ROOT, "smith-waterman-fpga-module_b200", "libsw_b200_check.so")
    if not os.path.exists(lib):
        pytest.skip("libsw_b200_check.so not built (make -C csrc CHECK=1)")
    if pkg.is_check_build():
        pytest.skip("already running the check build")
    env = dict(os.environ, SW_B200_LIB=lib)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu",
                        "-k", "not bounds_check_build", "-p", "no:cacheprovider"], capture_output=True, text=True, env=env,
                       timeout=1500, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout
