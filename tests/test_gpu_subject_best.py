"""GPU tests of the per-subject best output (sw_set_subject_best / sw_fetch_subject_best / sw_fetch_db_subject_best):
for every subject its best query row, the best score and the runner-up score, reduced on the GPU.  Every case compares
with (M.max(0), M.argmax(0), np.sort(M, 0)[-2], or -1 with one row) of the oracle matrix M."""
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.test_gpu_hits import _ragged
from tests.test_gpu_parity import _mutate, _oracle_matrix, _rand
from tests.test_gpu_round2 import _overflow_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def _revcomp(s):
    return "".join(COMP[c] for c in reversed(s))


def _want_best(mat):
    rows, ns = mat.shape
    if ns == 0:
        return np.zeros(0, np.int32), np.zeros(0, np.uint32), np.zeros(0, np.int32)
    second = np.sort(mat, 0)[-2] if rows > 1 else np.full(ns, -1)
    return mat.max(0).astype(np.int32), mat.argmax(0).astype(np.uint32), second.astype(np.int32)


def _assert_best(got, mat, msg=""):
    want = _want_best(mat)
    assert got[0].dtype == np.int32 and got[1].dtype == np.uint32 and got[2].dtype == np.int32
    for name, g, w in zip(("best_score", "best_row", "second_score"), got, want):
        np.testing.assert_array_equal(g, w, err_msg=f"{name} {msg}")


@pytest.mark.parametrize("choice", ["auto", "strip_s16x2_R25x2_G1", "strip_s16x2_R25x2_G1_U4_F31", "strip_s16x2_R16x1_G32",
                                    "strip_s16x2_R38x1_G4"])
def test_subject_best_every_variant_vs_oracle(oracle_mod, pkg, choice):
    rng = random.Random(41)
    queries = [_rand(rng, n) for n in (150, 40, 151, 300, 75)]
    subjects = _ragged(rng, queries, 3000)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        if choice != "auto":
            e.set_kernel_name(choice)
        e.set_queries(queries)
        e.set_subject_best(True)
        e.load_db(subjects)
        e.score_db()
        _assert_best(e.fetch_db_subject_best(), want, f"{choice} resident")
        e.score_batch(subjects)
        _assert_best(e.fetch_subject_best(), want, f"{choice} streaming")
        assert e.device_error_bits == 0


def test_subject_best_ties_and_one_row(oracle_mod, pkg):
    """Duplicated queries tie exactly: best_row is the lowest of the tied rows and second == best.  One query:
    second == -1 everywhere, zero-length subjects give (0, 0, -1)."""
    rng = random.Random(8)
    a, b, c = _rand(rng, 150), _rand(rng, 90), _rand(rng, 150)
    queries = [c, a, b, a, c, b]
    subjects = _ragged(rng, [a, b, c], 2500)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_subject_best(True)
        e.set_queries(queries)
        e.score_batch(subjects)
        got = e.fetch_subject_best()
    _assert_best(got, want, "duplicated queries")
    assert (got[2] == got[0]).all()                   # every row has a twin
    assert set(np.unique(got[1]).tolist()) <= {0, 1, 2}
    want1 = want[1:2]
    with pkg.Engine() as e:
        e.set_subject_best(True)
        e.set_queries([a])
        e.score_batch(subjects)
        got = e.fetch_subject_best()
    _assert_best(got, want1, "one row")
    assert (got[2] == -1).all() and (got[1] == 0).all()
    empty = np.array([len(s) == 0 for s in subjects])
    assert empty.any() and (got[0][empty] == 0).all()


def test_subject_best_streaming_and_shards(oracle_mod, pkg):
    """Two batches in flight (one empty, one of 3 subjects), ids through fetch_ids; a handle whose database is
    split over three shards of one GPU, and over every GPU plus a repeated one."""
    rng = random.Random(78)
    queries = [_rand(rng, 120), _rand(rng, 33), _rand(rng, 120)]
    batches = [_ragged(rng, queries, n) for n in (900, 3, 0, 450, 2001)]
    wants = [_oracle_matrix(oracle_mod, pkg, queries, b) if b else np.zeros((3, 0), np.int32) for b in batches]
    for gpu_ids in ([0, 0, 0], list(range(pkg.device_count())) + [0]):
        with pkg.Engine(gpu_ids=gpu_ids) as e:
            e.set_subject_best(True)
            e.set_queries(queries)
            got, ids = [], []
            e.score_batch(batches[0], ids=np.arange(len(batches[0]), dtype=np.uint64) + 1000)
            for k, b in enumerate(batches[1:], 1):
                e.score_batch(b, ids=np.arange(len(b), dtype=np.uint64) + 1000 * (k + 1))
                assert e.batches_in_flight == 2
                got.append(e.fetch_subject_best())
                ids.append(e.fetch_ids())
            got.append(e.fetch_subject_best())
            ids.append(e.fetch_ids())
            assert e.device_error_bits == 0
        for k, (b, g, w) in enumerate(zip(batches, got, wants)):
            _assert_best(g, w, str((gpu_ids, len(b))))
            assert ids[k].tolist() == list(range(1000 * (k + 1), 1000 * (k + 1) + len(b)))


@pytest.mark.parametrize("wave32", [True, False])
def test_subject_best_with_scores_beyond_16_bits(oracle_mod, pkg, wave32):
    """Pairs whose score leaves the 16-bit range update their subject from the exact 32-bit score (overflow list),
    exactly once: the best is exact (33 500) and the runner-up is the other row's score."""
    rng = random.Random(5)
    s, subjects = _overflow_case(rng)
    queries = [s, _rand(rng, 150), s[:6560]]
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    assert want[0, 0] == 33500 and want[2, 0] > 32767
    # wave mode 1: the long queries run on the band-pipelined kernel (sentinel in its scratch row); wave mode 0: on
    # the strip kernel, whose epilogue must leave the flagged pairs to the overflow list
    for wave in (1, 0):
        with pkg.Engine() as e:
            e.set_overflow_wave(wave32)
            e.set_wave_mode(wave)
            e.set_queries(queries)
            e.set_subject_best(True)
            e.score_batch(subjects)
            got = e.fetch_subject_best()
            assert ("wave" in e.last_kernel_name) == (wave == 1), e.last_kernel_name
            _assert_best(got, want, f"wave32={wave32} wave={wave}")
            assert got[0][0] == 33500 and got[1][0] == 0
            assert e.device_error_bits == 0


@pytest.mark.parametrize("sticky", ["-1", "0"])
def test_subject_best_band_pipelined_and_pass_split(oracle_mod, pkg, monkeypatch, sticky):
    """Queries on the band-pipelined kernel (a scratch score row per query, reduced by sbest_row_kernel), forced and
    automatic, next to a short query on the strip kernel; long queries with the pass split forced to 3 and to 64
    parts.  A (subject, row) pair that arrived twice would set second == best where the matrix says otherwise."""
    monkeypatch.setenv("SW_B200_STICKY", sticky)
    rng = random.Random(407)
    q1, q2, q3 = _rand(rng, 3000), _rand(rng, 1100), _rand(rng, 90)
    subjects = [q1[100:2900], _mutate(rng, q1, 0.05, 0.02), _rand(rng, 3000), "", _mutate(rng, q2, 0.1, 0.05), q2[500:1000],
                _rand(rng, 40), q3 + _rand(rng, 200), _mutate(rng, q1[1000:2500], 0.02, 0.01)]
    subjects += [_rand(rng, rng.randint(1, 900)) for _ in range(40)]
    want = _oracle_matrix(oracle_mod, pkg, [q1, q2, q3], subjects)
    for mode in (2, 1):
        with pkg.Engine() as e:
            e.set_wave_mode(mode)
            e.set_queries([q1, q2, q3])
            e.set_subject_best(True)
            e.score_batch(subjects)
            got = e.fetch_subject_best()
            assert "wave" in e.last_kernel_name, e.last_kernel_name
            _assert_best(got, want, f"wave mode {mode}")
            assert e.device_error_bits == 0
    # pass split: multi-chunk queries of equal length, ragged subjects with planted homologs
    queries = [_rand(rng, 1500), _rand(rng, 1500), _rand(rng, 1500)]
    subjects = []
    for _ in range(2500):
        if rng.random() < 0.2:
            q = rng.choice(queries)
            a = rng.randint(0, 1400)
            subjects.append(_mutate(rng, q[a:a + rng.randint(40, 500)], 0.06, 0.04) or "A")
        else:
            subjects.append(_rand(rng, rng.randint(0, 420)))
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    assert (np.sort(want, 0)[-2] < want.max(0)).sum() > 100
    for parts in (3, 64):
        with pkg.Engine() as e:
            e.set_wave_mode(0)
            e.set_kernel_name("strip_s16x2_R25x2_G1")
            e.set_pass_split(parts)
            e.set_subject_best(True)
            e.set_queries(queries)
            e.score_batch(subjects)
            got = e.fetch_subject_best()
            assert e.last_pass_parts >= 2
            assert e.device_error_bits == 0
        _assert_best(got, want, f"pass split {parts}")


def test_subject_best_score_width_strands_and_penalties(oracle_mod, pkg):
    """The RTL's 12-bit machine; both strands (rows 0 .. 2 nq - 1), with a palindromic query whose rows i and nq + i
    tie; a penalty set that is not compiled in (run-time specialised instance when NVRTC works)."""
    rng = random.Random(13)
    half = _rand(rng, 75)
    queries = [_rand(rng, 150), half + _revcomp(half), _rand(rng, 64)]
    subjects = _ragged(rng, queries, 2000)
    want12 = _oracle_matrix(oracle_mod, pkg, queries, subjects, score_width=12)
    with pkg.Engine(score_width=12) as e:
        e.set_subject_best(True)
        e.set_queries(queries)
        e.score_batch(subjects)
        _assert_best(e.fetch_subject_best(), want12, "w12")
    rc = [_revcomp(q) for q in queries]
    want2 = _oracle_matrix(oracle_mod, pkg, queries + rc, subjects)
    assert (want2[1] == want2[4]).all()
    with pkg.Engine() as e:
        e.set_strands(True)
        e.set_subject_best(True)
        e.set_queries(queries)
        e.score_batch(subjects)
        got = e.fetch_subject_best()
    _assert_best(got, want2, "both strands")
    assert not (got[1] == 4).any()                     # row 4 ties with row 1 and never wins
    params = dict(match=4, mismatch=-3, gap_open=-7, gap_extend=-3)
    wantp = _oracle_matrix(oracle_mod, pkg, queries, subjects, **params)
    ok, _msg = pkg.jit_compile_check("strip_s16x2_R25x2_G1", -7, -3)
    with pkg.Engine(**params) as e:
        e.set_jit(2 if ok == 1 else 0)
        e.set_subject_best(True)
        e.set_queries(queries)
        e.score_batch(subjects)
        got = e.fetch_subject_best()
        assert ok != 1 or "+jit" in e.last_kernel_name, e.last_kernel_name
        _assert_best(got, wantp, "penalties")


def _raises(pkg, code, fn):
    with pytest.raises(pkg.SwError) as ei:
        fn()
    assert ei.value.code == code


def test_subject_best_contract(oracle_mod, pkg):
    lib = pkg.load_library()
    rng = random.Random(4)
    queries = [_rand(rng, 150), _rand(rng, 80)]
    subjects = _ragged(rng, queries, 2000)
    ns = len(subjects)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_queries(queries)
        e.set_subject_best(True)
        # too small a cap: SW_ECAPACITY, nothing written, the batch stays; the retry returns the same result
        e.score_batch(subjects)
        bs = np.full(ns, 7, np.int32)
        br = np.full(ns, 7, np.uint32)
        sec = np.full(ns, 7, np.int32)
        assert lib.sw_fetch_subject_best(e.h, bs.ctypes.data, br.ctypes.data, sec.ctypes.data, ns - 1, -1) == pkg.SW_ECAPACITY
        assert e.batches_in_flight == 1 and (bs == 7).all() and (br == 7).all() and (sec == 7).all()
        launches = e.kernel_launches
        _assert_best(e.fetch_subject_best(), want, "retry")
        assert e.kernel_launches == launches                    # no rescoring
        # second_score = NULL
        e.score_batch(subjects)
        assert lib.sw_fetch_subject_best(e.h, bs.ctypes.data, br.ctypes.data, None, ns, -1) == pkg.SW_OK
        e._batch_ns.pop(0)
        w = _want_best(want)
        np.testing.assert_array_equal(bs, w[0])
        np.testing.assert_array_equal(br, w[1])
        assert (sec == 7).all()
        # the mode excludes top-k and hits, either way round
        _raises(pkg, pkg.SW_EINVAL, lambda: e.set_topk(4))
        _raises(pkg, pkg.SW_EINVAL, lambda: e.set_hits(30))
        e.set_subject_best(False)
        e.set_topk(4)
        _raises(pkg, pkg.SW_EINVAL, lambda: e.set_subject_best(True))
        e.set_topk(0)
        e.set_hits(30)
        _raises(pkg, pkg.SW_EINVAL, lambda: e.set_subject_best(True))
        e.set_hits(0)
        # SW_EAGAIN while a batch is in flight
        e.set_subject_best(True)
        e.score_batch(subjects)
        _raises(pkg, pkg.SW_EAGAIN, lambda: e.set_subject_best(False))
        # matrix / top-k / hits fetches of a subject-best batch: SW_ESTATE, the batch stays
        for fn in (lambda: e.fetch(), lambda: e.fetch_topk(), lambda: e.fetch_hits()):
            _raises(pkg, pkg.SW_ESTATE, fn)
        assert e.batches_in_flight == 1
        _assert_best(e.fetch_subject_best(), want, "after the refused fetches")
        e.load_db(subjects)
        e.score_db()
        for fn in (lambda: e.fetch_db(), lambda: e.fetch_best(), lambda: e.fetch_db_topk(), lambda: e.fetch_db_hits()):
            _raises(pkg, pkg.SW_ESTATE, fn)
        _assert_best(e.fetch_db_subject_best(), want, "resident")
        # the other way round: batches of the matrix, top-k and hits modes are not subject-best batches
        e.set_subject_best(False)
        for setup, drain in ((lambda: None, lambda: e.fetch()), (lambda: e.set_topk(4), lambda: e.fetch_topk()),
                             (lambda: e.set_hits(30), lambda: e.fetch_hits())):
            setup()
            e.score_batch(subjects)
            _raises(pkg, pkg.SW_ESTATE, lambda: e.fetch_subject_best())
            assert e.batches_in_flight == 1
            drain()
            e.set_topk(0)
            e.set_hits(0)
        e.load_db(subjects)
        e.score_db()
        _raises(pkg, pkg.SW_ESTATE, lambda: e.fetch_db_subject_best())
        # back to matrices: bit-identical to a handle that never used the mode
        e.score_batch(subjects)
        np.testing.assert_array_equal(e.fetch(), want)
        e.load_db(subjects)
        e.score_db()
        np.testing.assert_array_equal(e.fetch_db(), want)
        # the forced 32-bit scorer: refused at submit, nothing enqueued; the handle still scores
        e.set_kernel_choice(0, 0, True)
        e.set_subject_best(True)
        launches = e.kernel_launches
        _raises(pkg, pkg.SW_EINVAL, lambda: e.score_batch(subjects))
        e._batch_ns.clear()
        assert e.batches_in_flight == 0 and e.kernel_launches == launches
        assert lib.sw_score_db(e.h) == pkg.SW_EINVAL
        e.set_subject_best(False)
        np.testing.assert_array_equal(e.score(queries, subjects), want)
        assert e.last_kernel_name == "generic32"
        assert e.device_error_bits == 0
    with pkg.Engine() as e:
        np.testing.assert_array_equal(e.score(queries, subjects), want)


def test_subject_best_large_job_with_autotune(pkg):
    """A job large enough for the autotuner (>= 0.4 s of estimated work): its sample launches update nothing, so
    the result equals the argmax / runner-up of the same handle's int32 matrix."""
    q = pkg.random_packed_db(100, 150, seed=91)
    db = pkg.random_packed_db(1_200_000, 150, seed=92)
    pkg.plant_homologs(db, q, 0.01, seed=93)
    with pkg.Engine() as e:
        e.set_queries(q)
        e.load_db(db)
        e.score_db()
        mat = e.fetch_db()
        e.set_subject_best(True)
        e.set_autotune(True)                                    # forget the matrix mode's decision: tune again
        e.score_db()
        got = e.fetch_db_subject_best()
        assert e.device_error_bits == 0
    _assert_best(got, mat, "autotune")
    assert (got[0] > got[2]).sum() > 10000


def test_subject_best_golden_and_cli(golden, pkg, tmp_path):
    """query100.fa x data500.fa (a batch the latency path takes in matrix mode) equals the RTL's scores, row 0,
    runner-up -1; the CLI's -B output with the query twice: row 0 wins the tie, second == best."""
    q = golden["fasta"]["query100.fa"][0][1]
    db = golden["fasta"]["data500.fa"]
    rtl = [x for x in golden["rtl"] if x["file"] == "data500.fa_query100.fa_out.txt"][0]["rows"]
    score_of = {n: s for n, s, _t in rtl}
    names = [n for n, _ in db]
    want = [score_of[n] for n in names]
    with pkg.Engine() as e:
        e.set_subject_best(True)
        e.set_queries([q])
        e.score_batch([s for _, s in db])
        assert "+direct" not in e.last_kernel_name
        bs, br, sec = e.fetch_subject_best()
    assert bs.tolist() == want and (br == 0).all() and (sec == -1).all()
    cli = os.path.join(ROOT, "bin", "sw_b200_cli")
    qf, lf = tmp_path / "query100.fa", tmp_path / "data500.fa"
    qf.write_text(">query\n" + q + "\n>again\n" + q + "\n")
    lf.write_text("".join(f">{n}\n{s}\n" for n, s in db))
    r = subprocess.run([cli, "-q", str(qf), "-l", str(lf), "-t", "30", "-B"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    got = []
    for line in r.stdout.splitlines():
        m = re.match(r"(\S+) best (\S+) result: (-?\d+), second: (-?\d+)$", line)
        assert m, line
        assert m.group(2) == "query" and m.group(3) == m.group(4)
        got.append((m.group(1), int(m.group(3))))
    assert got == list(zip(names, want))
    for extra in (["-o", str(tmp_path / "o.txt")], ["-R", str(tmp_path / "r.txt")], ["-T", "10"]):
        r = subprocess.run([cli, "-q", str(qf), "-l", str(lf), "-B"] + extra, capture_output=True, text=True)
        assert r.returncode != 0 and "does not combine" in r.stdout


def test_subject_best_on_the_bounds_check_build(pkg):
    """This file again on libsw_b200_check.so (device-side index checks incl. the per-subject stores, canaries)."""
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

