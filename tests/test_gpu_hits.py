"""GPU tests of the hit-list output (sw_set_hits / sw_fetch_hits / sw_fetch_db_hits): every (row, subject)
pair scoring at least T, collected on the GPU -- the bank's (IDs, results, vld) stream (ScoreBank_v2.v:39-41)
filtered on `results`.  Every case compares with np.nonzero(want >= T) of the oracle matrix: same rows, same
indices, same scores, same (row-major) order."""
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


def _want_hits(mat, t):
    r, i = np.nonzero(mat >= t)
    return r.astype(np.uint32), i.astype(np.uint64), mat[r, i].astype(np.int32)


def _assert_hits(got, mat, t, msg=""):
    want = _want_hits(mat, t)
    assert got[0].dtype == np.uint32 and got[1].dtype == np.uint64 and got[2].dtype == np.int32
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w, err_msg=f"T={t} {msg}")


def _ragged(rng, queries, n):
    """0-260 nt subjects with empties, exact duplicates and mutated homologs of the queries."""
    subjects = []
    for _ in range(n):
        r = rng.random()
        if r < 0.15:
            subjects.append(_mutate(rng, rng.choice(queries), 0.1, 0.05)[:260])
        elif r < 0.25 and subjects:
            subjects.append(rng.choice(subjects))
        elif r < 0.28:
            subjects.append("")
        else:
            subjects.append(_rand(rng, rng.randint(1, 260)))
    return subjects


@pytest.mark.parametrize("choice", ["auto", "strip_s16x2_R25x2_G1", "strip_s16x2_R25x2_G1_U4_F31", "strip_s16x2_R16x1_G32",
                                    "strip_s16x2_R38x1_G4"])
def test_hits_every_variant_vs_oracle(oracle_mod, pkg, choice):
    rng = random.Random(31)
    queries = [_rand(rng, n) for n in (150, 40, 151, 300, 75)]
    subjects = _ragged(rng, queries, 3000)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    top = int(want.max())
    with pkg.Engine() as e:
        if choice != "auto":
            e.set_kernel_name(choice)
        e.set_queries(queries)
        for t in (1, top // 3, top, top + 1):
            e.set_hits(t, 20000)
            e.load_db(subjects)
            e.score_db()
            got = e.fetch_db_hits()
            _assert_hits(got, want, t, f"{choice} resident")
            e.score_batch(subjects)
            _assert_hits(e.fetch_hits(), want, t, f"{choice} streaming")
            if t == top + 1:
                assert got[0].size == 0
        assert e.device_error_bits == 0


def test_hits_streaming_and_shards(oracle_mod, pkg):
    """Two batches in flight (one empty, one of 3 subjects), ids through fetch_ids; a handle whose database is
    split over three shards of one GPU, and over every GPU plus a repeated one."""
    rng = random.Random(77)
    queries = [_rand(rng, 120), _rand(rng, 33)]
    batches = [_ragged(rng, queries, n) for n in (900, 3, 0, 450, 2001)]
    wants = [_oracle_matrix(oracle_mod, pkg, queries, b) if b else np.zeros((2, 0), np.int32) for b in batches]
    t = 40
    for gpu_ids in ([0, 0, 0], list(range(pkg.device_count())) + [0]):
        with pkg.Engine(gpu_ids=gpu_ids) as e:
            e.set_hits(t, 5000)
            e.set_queries(queries)
            got, ids = [], []
            e.score_batch(batches[0], ids=np.arange(len(batches[0]), dtype=np.uint64) + 1000)
            for k, b in enumerate(batches[1:], 1):
                e.score_batch(b, ids=np.arange(len(b), dtype=np.uint64) + 1000 * (k + 1))
                assert e.batches_in_flight == 2
                got.append(e.fetch_hits())
                ids.append(e.fetch_ids())
            got.append(e.fetch_hits())
            ids.append(e.fetch_ids())
            assert e.device_error_bits == 0
        for k, (b, g, w) in enumerate(zip(batches, got, wants)):
            _assert_hits(g, w, t, str((gpu_ids, len(b))))
            assert ids[k].tolist() == list(range(1000 * (k + 1), 1000 * (k + 1) + len(b)))


@pytest.mark.parametrize("wave32", [True, False])
def test_hits_with_scores_beyond_16_bits(oracle_mod, pkg, wave32):
    """Pairs whose score leaves the 16-bit range reach the list from their exact 32-bit score (overflow list),
    never twice: T below and above 32 767, with the 32-bit band scorer and with the one-thread scorer."""
    rng = random.Random(5)
    s, subjects = _overflow_case(rng)
    queries = [s, _rand(rng, 150)]
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    assert want[0, 0] == 33500
    # wave mode 1: the long query runs on the band-pipelined kernel (sentinel in its scratch row); wave mode 0: on
    # the strip kernel, whose epilogue must leave the flagged pairs to the overflow list
    for wave in (1, 0):
        with pkg.Engine() as e:
            e.set_overflow_wave(wave32)
            e.set_wave_mode(wave)
            e.set_queries(queries)
            for t in (1, 30000, 32767, 33000):
                e.set_hits(t, 1000)
                e.score_batch(subjects)
                got = e.fetch_hits()
                assert ("wave" in e.last_kernel_name) == (wave == 1), e.last_kernel_name
                _assert_hits(got, want, t, f"wave32={wave32} wave={wave}")
            assert e.device_error_bits == 0


@pytest.mark.parametrize("sticky", ["-1", "0"])
def test_hits_band_pipelined_and_pass_split(oracle_mod, pkg, monkeypatch, sticky):
    """Queries on the band-pipelined kernel (a scratch score row per query, filtered by hits_row_kernel), forced
    and automatic, next to a short query on the strip kernel; long queries with the pass split forced to 3
    parts; two work orders."""
    monkeypatch.setenv("SW_B200_STICKY", sticky)
    rng = random.Random(406)
    q1, q2, q3 = _rand(rng, 3000), _rand(rng, 1100), _rand(rng, 90)
    subjects = [q1[100:2900], _mutate(rng, q1, 0.05, 0.02), _rand(rng, 3000), "", _mutate(rng, q2, 0.1, 0.05), q2[500:1000],
                _rand(rng, 40), q3 + _rand(rng, 200), _mutate(rng, q1[1000:2500], 0.02, 0.01)]
    subjects += [_rand(rng, rng.randint(1, 900)) for _ in range(40)]
    want = _oracle_matrix(oracle_mod, pkg, [q1, q2, q3], subjects)
    for mode in (2, 1):
        with pkg.Engine() as e:
            e.set_wave_mode(mode)
            e.set_queries([q1, q2, q3])
            for t in (1, 100, 5000):
                e.set_hits(t, 1000)
                e.score_batch(subjects)
                got = e.fetch_hits()
                assert "wave" in e.last_kernel_name, e.last_kernel_name
                _assert_hits(got, want, t, f"wave mode {mode}")
            assert e.device_error_bits == 0
    # pass split: multi-chunk queries of equal length, ragged subjects with planted homologs
    queries = [_rand(rng, 1500), _rand(rng, 1500)]
    subjects = []
    for _ in range(2500):
        if rng.random() < 0.2:
            q = rng.choice(queries)
            a = rng.randint(0, 1400)
            subjects.append(_mutate(rng, q[a:a + rng.randint(40, 500)], 0.06, 0.04) or "A")
        else:
            subjects.append(_rand(rng, rng.randint(0, 420)))
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    with pkg.Engine() as e:
        e.set_wave_mode(0)
        e.set_kernel_name("strip_s16x2_R25x2_G1")
        e.set_pass_split(3)
        e.set_hits(60, 20000)
        e.set_queries(queries)
        e.score_batch(subjects)
        got = e.fetch_hits()
        assert e.last_pass_parts >= 2
        assert e.device_error_bits == 0
    _assert_hits(got, want, 60, "pass split")


def test_hits_score_width_strands_and_penalties(oracle_mod, pkg):
    """The RTL's 12-bit machine; both strands (rows 0 .. 2 nq - 1); a penalty set that is not compiled in
    (run-time specialised instance when NVRTC works, else the run-time-operand instance)."""
    rng = random.Random(12)
    queries = [_rand(rng, 150), _rand(rng, 64)]
    subjects = _ragged(rng, queries, 2000)
    want12 = _oracle_matrix(oracle_mod, pkg, queries, subjects, score_width=12)
    with pkg.Engine(score_width=12) as e:
        e.set_hits(30, 10000)
        e.set_queries(queries)
        e.score_batch(subjects)
        _assert_hits(e.fetch_hits(), want12, 30, "w12")
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    rc = ["".join(comp[c] for c in reversed(q)) for q in queries]
    want2 = _oracle_matrix(oracle_mod, pkg, queries + rc, subjects)
    with pkg.Engine() as e:
        e.set_strands(True)
        e.set_hits(35, 10000)
        e.set_queries(queries)
        e.score_batch(subjects)
        _assert_hits(e.fetch_hits(), want2, 35, "both strands")
    params = dict(match=4, mismatch=-3, gap_open=-7, gap_extend=-3)
    wantp = _oracle_matrix(oracle_mod, pkg, queries, subjects, **params)
    ok, _msg = pkg.jit_compile_check("strip_s16x2_R25x2_G1", -7, -3)
    with pkg.Engine(**params) as e:
        e.set_jit(2 if ok == 1 else 0)
        e.set_hits(25, 10000)
        e.set_queries(queries)
        e.score_batch(subjects)
        got = e.fetch_hits()
        assert ok != 1 or "+jit" in e.last_kernel_name, e.last_kernel_name
        _assert_hits(got, wantp, 25, "penalties")


def test_hits_contract(oracle_mod, pkg):
    lib = pkg.load_library()
    rng = random.Random(3)
    queries = [_rand(rng, 150), _rand(rng, 80)]
    subjects = _ragged(rng, queries, 2000)
    want = _oracle_matrix(oracle_mod, pkg, queries, subjects)
    t = 30
    n = int((want >= t).sum())
    assert n > 20
    import ctypes as C
    with pkg.Engine() as e:
        e.set_queries(queries)
        # max_hits below the total: SW_ERANGE with the exact count, and the batch is consumed
        e.set_hits(t, n // 2)
        e.score_batch(subjects)
        cnt = C.c_size_t(0)
        assert lib.sw_fetch_hits(e.h, None, None, None, 0, C.byref(cnt), -1) == pkg.SW_ERANGE
        assert cnt.value == n and e.batches_in_flight == 0
        e._batch_ns.clear()
        # too small a cap: SW_ECAPACITY, nothing written, the retry returns the identical list
        e.set_hits(t, n)
        e.score_batch(subjects)
        row = np.full(n - 1, 7, np.uint32)
        idx = np.full(n - 1, 7, np.uint64)
        sc = np.full(n - 1, 7, np.int32)
        assert lib.sw_fetch_hits(e.h, row.ctypes.data, idx.ctypes.data, sc.ctypes.data, n - 1, C.byref(cnt), -1) == pkg.SW_ECAPACITY
        assert cnt.value == n and e.batches_in_flight == 1
        launches = e.kernel_launches
        assert (row == 7).all() and (idx == 7).all() and (sc == 7).all()
        got = e.fetch_hits()
        assert e.kernel_launches == launches                    # no rescoring, no second sort
        _assert_hits(got, want, t)
        # hits and top-k exclude each other
        with pytest.raises(pkg.SwError) as ei:
            e.set_topk(4)
        assert ei.value.code == pkg.SW_EINVAL
        e.set_hits(0)
        e.set_topk(4)
        with pytest.raises(pkg.SwError) as ei:
            e.set_hits(t)
        assert ei.value.code == pkg.SW_EINVAL
        e.set_topk(0)
        assert lib.sw_set_hits(e.h, -1, 10) == pkg.SW_EINVAL and lib.sw_set_hits(e.h, 5, 0) == pkg.SW_EINVAL
        # mode mismatches: SW_ESTATE, the batch stays
        e.set_hits(t, n)
        e.score_batch(subjects)
        for fn in (lambda: e.fetch(), lambda: e.fetch_topk()):
            with pytest.raises(pkg.SwError) as ei:
                fn()
            assert ei.value.code == pkg.SW_ESTATE
        assert e.batches_in_flight == 1
        _assert_hits(e.fetch_hits(), want, t)
        e.load_db(subjects)
        e.score_db()
        for fn in (lambda: e.fetch_db(), lambda: e.fetch_best(), lambda: e.fetch_db_topk()):
            with pytest.raises(pkg.SwError) as ei:
                fn()
            assert ei.value.code == pkg.SW_ESTATE
        _assert_hits(e.fetch_db_hits(), want, t)
        e.set_hits(0)
        e.score_batch(subjects)
        with pytest.raises(pkg.SwError) as ei:
            e.fetch_hits()
        assert ei.value.code == pkg.SW_ESTATE
        # back to matrices: bit-identical to a handle that never used hits
        np.testing.assert_array_equal(e.fetch(), want)
        e.load_db(subjects)                                     # (the small batch above took the resident slot)
        e.score_db()
        np.testing.assert_array_equal(e.fetch_db(), want)
        # the forced 32-bit scorer and hits: refused at submit, nothing enqueued; the handle still scores
        e.set_kernel_choice(0, 0, True)
        e.set_hits(t, n)
        launches = e.kernel_launches
        with pytest.raises(pkg.SwError) as ei:
            e.score_batch(subjects)
        assert ei.value.code == pkg.SW_EINVAL
        e._batch_ns.clear()
        assert e.batches_in_flight == 0 and e.kernel_launches == launches
        assert lib.sw_score_db(e.h) == pkg.SW_EINVAL
        e.set_hits(0)
        np.testing.assert_array_equal(e.score(queries, subjects), want)
        assert e.last_kernel_name == "generic32"
        assert e.device_error_bits == 0


def test_hits_large_job_with_autotune(pkg):
    """A job large enough for the autotuner (>= 0.4 s of estimated work): its sample launches append nothing,
    so the list equals the same handle's int32 matrix filtered on the host and holds every pair once."""
    q = pkg.random_packed_db(100, 150, seed=91)
    db = pkg.random_packed_db(1_200_000, 150, seed=92)
    pkg.plant_homologs(db, q, 0.01, seed=93)
    t = 100
    with pkg.Engine() as e:
        e.set_queries(q)
        e.load_db(db)
        e.score_db()
        mat = e.fetch_db()
        e.set_hits(t, 1 << 20)
        e.set_autotune(True)                                    # forget the matrix mode's decision: tune again
        e.score_db()
        got = e.fetch_db_hits()
        assert e.device_error_bits == 0
    assert got[0].size > 5000
    _assert_hits(got, mat, t, "autotune")
    key = got[0].astype(np.uint64) * np.uint64(1_200_000) + got[1]
    assert np.unique(key).size == key.size


def test_hits_golden_and_cli(golden, pkg, tmp_path):
    """query100.fa x data500.fa (a batch the latency path takes in matrix mode) in hits mode equals the RTL's
    scores filtered at T; so does the CLI's -T output."""
    q = golden["fasta"]["query100.fa"][0][1]
    db = golden["fasta"]["data500.fa"]
    rtl = [x for x in golden["rtl"] if x["file"] == "data500.fa_query100.fa_out.txt"][0]["rows"]
    score_of = {n: s for n, s, _t in rtl}
    t = sorted(score_of.values())[len(score_of) * 3 // 4]
    names = [n for n, _ in db]
    want = sorted((names.index(n), s) for n, s in score_of.items() if s >= t)
    assert 10 < len(want) < len(names)
    with pkg.Engine() as e:
        e.set_hits(t, 1000)
        e.set_queries([q])
        e.score_batch([s for _, s in db])
        assert "+direct" not in e.last_kernel_name
        row, idx, sc = e.fetch_hits()
    assert (row == 0).all()
    assert list(zip(idx.tolist(), sc.tolist())) == want
    cli = os.path.join(ROOT, "bin", "sw_b200_cli")
    qf, lf = tmp_path / "query100.fa", tmp_path / "data500.fa"
    qf.write_text(">query\n" + q + "\n")
    lf.write_text("".join(f">{n}\n{s}\n" for n, s in db))
    r = subprocess.run([cli, "-q", str(qf), "-l", str(lf), "-t", "30", "-T", str(t)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    got = []
    for line in r.stdout.splitlines():
        m = re.match(r"query x (\S+) result: (-?\d+), biased: (\d+)\(0x([0-9a-f]{4})\)$", line)
        assert m, line
        assert int(m.group(3)) == int(m.group(2)) + 2048 == int(m.group(4), 16)
        got.append((names.index(m.group(1)), int(m.group(2))))
    assert got == want
    r = subprocess.run([cli, "-q", str(qf), "-l", str(lf), "-T", str(t), "-o", str(tmp_path / "o.txt")], capture_output=True, text=True)
    assert r.returncode != 0 and "does not combine" in r.stdout


def test_hits_on_the_bounds_check_build(pkg):
    """This file again on libsw_b200_check.so (device-side index checks incl. the hit-list stores, canaries)."""
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
