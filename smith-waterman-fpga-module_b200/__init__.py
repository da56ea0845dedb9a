"""B200-native score-only Smith-Waterman engine -- Python plumbing over the C ABI.

The product is ``libsw_b200.so`` (hand-written CUDA for sm_100a behind the C ABI of
``include/sw_b200.h``).  This module only binds it with ctypes so that tests and
``bench.py`` can drive it; it contains no scoring code and no CPU fallback: if the
library is missing or no B200 is visible, construction raises.

Operator surface mirrored (reference: ScoreBank/ScoreBank_v2.v:31-44 and
capi_sample_aligner/software-C,C++/src/main_test.c:290-528):
    Engine(match, mismatch, gap_open, gap_extend)   <- ld_penalties / penalties bus
    Engine.set_queries(...)                          <- type-01 record, ld_q
    Engine.score_batch(...)                          <- stream of type-10 records
    Engine.fetch(timeout_ms)                         <- (IDs, results, vld) + WED poll, result-2048
    Engine.fetch_hits(timeout_ms)                    <- the same stream filtered on results >= min_score
    Engine.fetch_subject_best(timeout_ms)            <- per ID: the best query row, its score and the runner-up
"""
import ctypes as C
import os

import numpy as np

from .seqio import pack_sequences, plant_homologs, random_packed_db  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SW_B200_LIB", os.path.join(_HERE, "libsw_b200.so"))   # override: A/B builds

SW_OK, SW_EINVAL, SW_ENOMEM, SW_ECUDA, SW_ENODEV = 0, -1, -2, -3, -4
SW_ESTATE, SW_ETIMEOUT, SW_ECAPACITY, SW_EIO, SW_EAGAIN = -5, -6, -7, -8, -9
SW_ERANGE, SW_EDEVICE = -10, -11
SW_OUTPUT_I32, SW_OUTPUT_I16 = 0, 1


class SwParams(C.Structure):
    _fields_ = [("match", C.c_int16), ("mismatch", C.c_int16), ("gap_open", C.c_int16),
                ("gap_extend", C.c_int16), ("score_width", C.c_int32)]


class SwStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("load_ms", "enqueue_ms", "fetch_wait_ms", "fetch_drain_ms",
                                          "kernel_ms_max", "kernel_ms_min")]


class SwError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sw_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """Loads libsw_b200.so (built by ``__graft_entry__.build()`` / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). "
                          "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u64, sz, i32 = C.c_void_p, C.c_uint64, C.c_size_t, C.c_int
    L.sw_default_params.argtypes = [C.POINTER(SwParams)]
    L.sw_default_params.restype = None
    L.sw_init.argtypes = [C.POINTER(vp), C.POINTER(SwParams), C.POINTER(C.c_int), i32]
    L.sw_destroy.argtypes = [vp]
    L.sw_destroy.restype = None
    L.sw_set_queries.argtypes = [vp, vp, vp, vp, i32]
    L.sw_score_batch.argtypes = [vp, vp, vp, vp, vp, sz]
    L.sw_fetch.argtypes = [vp, vp, sz, i32]
    L.sw_fetch_ids.argtypes = [vp, vp, sz]
    L.sw_load_db.argtypes = [vp, vp, vp, vp, vp, sz]
    L.sw_score_db.argtypes = [vp]
    L.sw_wait.argtypes = [vp, i32]
    L.sw_fetch_db.argtypes = [vp, vp, sz]
    L.sw_fetch_best.argtypes = [vp, vp, vp, i32]
    L.sw_strerror.argtypes = [i32]
    L.sw_strerror.restype = C.c_char_p
    L.sw_last_cuda_error.argtypes = [vp]
    L.sw_last_cuda_error_string.argtypes = [vp]
    L.sw_last_cuda_error_string.restype = C.c_char_p
    L.sw_last_kernel_ms.argtypes = [vp]
    L.sw_last_kernel_ms.restype = C.c_double
    L.sw_kernel_launches.argtypes = [vp]
    L.sw_kernel_launches.restype = u64
    L.sw_last_cells.argtypes = [vp]
    L.sw_last_cells.restype = u64
    L.sw_last_kernel_name.argtypes = [vp]
    L.sw_last_kernel_name.restype = C.c_char_p
    L.sw_set_kernel_choice.argtypes = [vp, i32, i32, i32]
    L.sw_set_arith.argtypes = [vp, i32]
    L.sw_kernel_variant_count.restype = i32
    L.sw_kernel_variant_name.argtypes = [i32]
    L.sw_kernel_variant_name.restype = C.c_char_p
    L.sw_set_kernel_name.argtypes = [vp, C.c_char_p]
    L.sw_plan_shards.argtypes = [vp, sz, i32, vp]
    L.sw_set_fixed_penalty_kernels.argtypes = [i32]
    L.sw_set_autotune.argtypes = [vp, i32]
    L.sw_set_strands.argtypes = [vp, i32]
    L.sw_query_rows.argtypes = [vp]
    L.sw_batches_in_flight.argtypes = [vp]
    L.sw_set_output.argtypes = [vp, i32]
    L.sw_set_topk.argtypes = [vp, i32]
    L.sw_fetch_i16.argtypes = [vp, vp, sz, i32]
    L.sw_fetch_db_i16.argtypes = [vp, vp, sz]
    L.sw_fetch_overflow.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
    L.sw_fetch_topk.argtypes = [vp, vp, vp, sz, i32]
    L.sw_fetch_db_topk.argtypes = [vp, vp, vp, sz]
    L.sw_set_hits.argtypes = [vp, C.c_int32, sz]
    L.sw_fetch_hits.argtypes = [vp, vp, vp, vp, sz, C.POINTER(sz), i32]
    L.sw_fetch_db_hits.argtypes = [vp, vp, vp, vp, sz, C.POINTER(sz)]
    L.sw_set_subject_best.argtypes = [vp, i32]
    L.sw_fetch_subject_best.argtypes = [vp, vp, vp, vp, sz, i32]
    L.sw_fetch_db_subject_best.argtypes = [vp, vp, vp, vp, sz]
    L.sw_locate_db.argtypes = [vp, vp, vp, sz, vp, vp]
    L.sw_align_db.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, sz, vp]
    L.sw_device_error_bits.argtypes = [vp]
    L.sw_device_error_bits.restype = C.c_uint
    L.sw_is_check_build.restype = i32
    L.sw_set_jit.argtypes = [vp, i32]
    L.sw_jit_is_available.restype = i32
    L.sw_jit_compile_check.argtypes = [C.c_char_p, i32, i32, C.c_char_p, sz]
    L.sw_set_small_batch_path.argtypes = [vp, i32]
    L.sw_set_small_batch_timing.argtypes = [vp, i32]
    L.sw_set_wave_mode.argtypes = [vp, i32]
    L.sw_set_overflow_wave.argtypes = [vp, i32, C.c_ulonglong]
    L.sw_set_launch_plan.argtypes = [vp, i32, i32]
    L.sw_set_pass_split.argtypes = [vp, i32]
    L.sw_last_pass_parts.argtypes = [vp]
    L.sw_plan_pass_parts.argtypes = [i32, i32, C.c_ulonglong, i32, i32, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.sw_get_stats.argtypes = [vp, C.POINTER(SwStats)]
    L.sw_params_in_exact_domain.argtypes = [C.POINTER(SwParams)]
    L.sw_device_count.restype = i32
    L.sw_version.restype = C.c_char_p
    L.sw_pack_2bit.argtypes = [C.c_char_p, sz, vp]
    L.sw_pack_2bit.restype = None
    L.sw_unpack_2bit.argtypes = [vp, sz, C.c_char_p]
    L.sw_unpack_2bit.restype = None
    _lib = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data


class Engine:
    """One handle = one control thread; not re-entrant (like the reference host)."""

    def __init__(self, match=5, mismatch=-4, gap_open=-12, gap_extend=-4, score_width=0, gpu_ids=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        p = SwParams(match, mismatch, gap_open, gap_extend, score_width)
        if gpu_ids is None:
            rc = self.lib.sw_init(C.byref(self.h), C.byref(p), None, 0)
        else:
            arr = (C.c_int * len(gpu_ids))(*gpu_ids)
            rc = self.lib.sw_init(C.byref(self.h), C.byref(p), arr, len(gpu_ids))
        if rc != SW_OK:
            self.h = C.c_void_p()
            raise SwError(rc, self.lib.sw_strerror(rc).decode())
        self.nq = 0          # rows of the score matrix (queries x strands)
        self.ns = 0          # subjects of the resident database / last submitted batch
        self._batch_ns = []  # subjects of the batches in flight, oldest first
        self.out_mode = SW_OUTPUT_I32
        self.topk = 0
        self.hits = 0        # min_score of the hit-list mode (0 = off)
        self.subject_best = False
        self._ids_ns = 0     # subjects of the batch sw_fetch_ids refers to (last loaded / fetched)
        self._qlen = np.zeros(0, np.uint64)    # query lengths of set_queries (row nq + i has query i's length)
        self._db_len = np.zeros(0, np.uint64)  # subject lengths of load_db (align_db sizes its CIGAR buffer with both)

    # -- plumbing ---------------------------------------------------------------------
    def _check(self, rc):
        if rc != SW_OK:
            msg = self.lib.sw_strerror(rc).decode()
            if rc == SW_ECUDA:
                msg += " [" + self.lib.sw_last_cuda_error_string(self.h).decode() + "]"
            raise SwError(rc, msg)

    def close(self):
        if self.h:
            self.lib.sw_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @staticmethod
    def _as_packed(seqs):
        if isinstance(seqs, tuple):
            packed, ln, off = seqs
            return (np.ascontiguousarray(packed, dtype=np.uint8), np.ascontiguousarray(ln, dtype=np.uint32),
                    np.ascontiguousarray(off, dtype=np.uint64))
        return pack_sequences(seqs)

    # -- operator surface ---------------------------------------------------------------
    def set_strands(self, both):
        """both=True: also score the reverse complement of every query (rows nq..2nq-1)."""
        self._check(self.lib.sw_set_strands(self.h, int(bool(both))))

    def set_queries(self, queries):
        packed, ln, off = self._as_packed(queries)
        self._check(self.lib.sw_set_queries(self.h, _ptr(packed), _ptr(ln), _ptr(off), len(ln)))
        self.nq = int(self.lib.sw_query_rows(self.h))
        self._qlen = ln.astype(np.uint64)

    def score_batch(self, subjects, ids=None):
        packed, ln, off = self._as_packed(subjects)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint64)
        self._check(self.lib.sw_score_batch(self.h, _ptr(packed), _ptr(ln), _ptr(off), _ptr(ids_a), len(ln)))
        self.ns = len(ln)
        self._batch_ns.append(len(ln))

    def fetch(self, timeout_ms=-1, out=None):
        """Scores of the OLDEST batch in flight (two may be in flight): int32 or, after
        set_output(SW_OUTPUT_I16), int16 matrix [rows, ns]."""
        ns = self._batch_ns[0] if self._batch_ns else self.ns
        i16 = self.out_mode == SW_OUTPUT_I16
        if out is None:
            out = np.empty((self.nq, ns), dtype=np.int16 if i16 else np.int32)
        fn = self.lib.sw_fetch_i16 if i16 else self.lib.sw_fetch
        self._check(fn(self.h, _ptr(out), out.size, timeout_ms))
        if self._batch_ns:
            self._ids_ns = self._batch_ns.pop(0)
        return out

    def set_output(self, mode):
        """SW_OUTPUT_I32 (default) or SW_OUTPUT_I16 (half the HBM / D2H bytes; scores above 32767
        come back through fetch_overflow)."""
        self._check(self.lib.sw_set_output(self.h, mode))
        self.out_mode = mode

    def set_topk(self, k):
        """k > 0: fused per-query top-k, no score matrix (fetch_topk / fetch_db_topk); 0 = matrices."""
        self._check(self.lib.sw_set_topk(self.h, k))
        self.topk = k

    def fetch_overflow(self):
        """(flat index iq * ns + is, int32 score) of the scores above 32767 of the batch fetched last."""
        cnt = C.c_size_t(0)
        self._check(self.lib.sw_fetch_overflow(self.h, None, None, 0, C.byref(cnt)))
        idx = np.empty(cnt.value, dtype=np.uint64)
        sc = np.empty(cnt.value, dtype=np.int32)
        if cnt.value:
            self._check(self.lib.sw_fetch_overflow(self.h, _ptr(idx), _ptr(sc), cnt.value, C.byref(cnt)))
        return idx, sc

    def fetch_topk(self, timeout_ms=-1):
        """(scores [rows, k], index [rows, k]) of the oldest batch in flight; index = input index in the batch."""
        sc = np.empty((self.nq, self.topk), dtype=np.int32)
        ix = np.empty((self.nq, self.topk), dtype=np.uint64)
        self._check(self.lib.sw_fetch_topk(self.h, _ptr(sc), _ptr(ix), sc.size, timeout_ms))
        if self._batch_ns:
            self._ids_ns = self._batch_ns.pop(0)
        return sc, ix

    def fetch_db_topk(self):
        sc = np.empty((self.nq, self.topk), dtype=np.int32)
        ix = np.empty((self.nq, self.topk), dtype=np.uint64)
        self._check(self.lib.sw_fetch_db_topk(self.h, _ptr(sc), _ptr(ix), sc.size))
        return sc, ix

    def set_hits(self, min_score, max_hits=1 << 24):
        """min_score >= 1: instead of a matrix, list every (row, subject) pair scoring >= min_score
        (fetch_hits / fetch_db_hits); each GPU's list holds max_hits entries.  0 = back to matrices."""
        self._check(self.lib.sw_set_hits(self.h, int(min_score), int(max_hits)))
        self.hits = int(min_score)

    def _hits(self, call):
        cnt = C.c_size_t(0)
        rc = call(None, None, None, 0, C.byref(cnt))            # size query (SW_OK with no hits at all)
        row = np.empty(cnt.value if rc == SW_ECAPACITY else 0, dtype=np.uint32)
        idx = np.empty(row.size, dtype=np.uint64)
        sc = np.empty(row.size, dtype=np.int32)
        if rc == SW_ECAPACITY:
            rc = call(_ptr(row), _ptr(idx), _ptr(sc), row.size, C.byref(cnt))
        return rc, row, idx, sc

    def fetch_hits(self, timeout_ms=-1):
        """(row uint32, index uint64, score int32) of the oldest batch in flight: every entry of its int32
        matrix >= min_score, row-major order; index = input index in the batch."""
        rc, row, idx, sc = self._hits(lambda r, i, s, cap, cnt: self.lib.sw_fetch_hits(self.h, r, i, s, cap, cnt, timeout_ms))
        if self._batch_ns and rc in (SW_OK, SW_ERANGE):          # SW_ERANGE consumes the batch too
            self._ids_ns = self._batch_ns.pop(0)
        self._check(rc)
        return row, idx, sc

    def fetch_db_hits(self):
        """fetch_hits for the resident database (after score_db)."""
        rc, row, idx, sc = self._hits(lambda r, i, s, cap, cnt: self.lib.sw_fetch_db_hits(self.h, r, i, s, cap, cnt))
        self._check(rc)
        return row, idx, sc

    def set_subject_best(self, enable=True):
        """True: instead of a matrix, per subject its best row, best score and runner-up score
        (fetch_subject_best / fetch_db_subject_best).  False = back to matrices."""
        self._check(self.lib.sw_set_subject_best(self.h, int(bool(enable))))
        self.subject_best = bool(enable)

    @staticmethod
    def _subject_best_arrays(ns):
        return np.empty(ns, dtype=np.int32), np.empty(ns, dtype=np.uint32), np.empty(ns, dtype=np.int32)

    def fetch_subject_best(self, timeout_ms=-1):
        """(best_score int32[ns], best_row uint32[ns], second_score int32[ns]) of the oldest batch in flight:
        per subject (input order) the column maximum of its int32 matrix, the lowest row reaching it, and the
        largest score of the other rows (-1 with one row)."""
        ns = self._batch_ns[0] if self._batch_ns else self.ns
        bs, br, sec = self._subject_best_arrays(ns)
        rc = self.lib.sw_fetch_subject_best(self.h, _ptr(bs), _ptr(br), _ptr(sec), ns, timeout_ms)
        if self._batch_ns and rc in (SW_OK, SW_ERANGE):          # SW_ERANGE consumes the batch too
            self._ids_ns = self._batch_ns.pop(0)
        self._check(rc)
        return bs, br, sec

    def fetch_db_subject_best(self):
        """fetch_subject_best for the resident database (after score_db)."""
        bs, br, sec = self._subject_best_arrays(self.ns)
        self._check(self.lib.sw_fetch_db_subject_best(self.h, _ptr(bs), _ptr(br), _ptr(sec), self.ns))
        return bs, br, sec

    def locate_db(self, rows, index):
        """Where the best local alignment of each (query row, subject) pair of the resident database begins and
        ends: (score int32[n], coord uint32[n, 4]) with coord = (q_begin, q_end, s_begin, s_end), 0-based and
        half-open; index = input index in the database of load_db.  The tie rule is in include/sw_b200.h."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32).reshape(-1)
        index = np.ascontiguousarray(index, dtype=np.uint64).reshape(-1)
        if rows.size != index.size:
            raise ValueError("rows and index differ in length")
        score = np.empty(rows.size, dtype=np.int32)
        coord = np.empty((rows.size, 4), dtype=np.uint32)
        self._check(self.lib.sw_locate_db(self.h, _ptr(rows), _ptr(index), rows.size, _ptr(score), _ptr(coord)))
        return score, coord

    def align_db(self, rows, index):
        """The CIGAR of each pair's located alignment: (score int32[n], coord uint32[n, 4], cigar_off uint64[n + 1],
        cigar uint32[...]), with score and coord as locate_db gives them and pair i's BAM-encoded ops (len << 4 | op)
        in cigar[cigar_off[i]:cigar_off[i + 1]]; cigar_str turns them into text.  The walk's tie rules are in
        include/sw_b200.h.  One call: the buffer holds sum(row length + subject length), which always suffices."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32).reshape(-1)
        index = np.ascontiguousarray(index, dtype=np.uint64).reshape(-1)
        if rows.size != index.size:
            raise ValueError("rows and index differ in length")
        n = rows.size
        score = np.empty(n, dtype=np.int32)
        coord = np.empty((n, 4), dtype=np.uint32)
        cigar_off = np.empty(n + 1, dtype=np.uint64)
        cap = 0
        if n and self._qlen.size and self._db_len.size:
            # out-of-range rows or indices only mis-size the buffer: the library rejects them
            qlen = self._qlen[rows % self._qlen.size]
            slen = np.take(self._db_len, index.astype(np.int64), mode="clip")
            cap = int(qlen.sum(dtype=np.uint64)) + int(slen.sum(dtype=np.uint64))
        cigar = np.empty(cap, dtype=np.uint32)
        count = C.c_size_t(0)
        self._check(self.lib.sw_align_db(self.h, _ptr(rows), _ptr(index), n, _ptr(score), _ptr(coord), _ptr(cigar_off),
                                         _ptr(cigar) if cap else None, cap, C.byref(count)))
        return score, coord, cigar_off, cigar[:count.value]

    def set_jit(self, mode):
        self._check(self.lib.sw_set_jit(self.h, mode))

    def set_wave_mode(self, mode):
        """Band-pipelined kernel for few long pairs: 0 never, 1 automatic, 2 whenever possible."""
        self._check(self.lib.sw_set_wave_mode(self.h, mode))

    def set_overflow_wave(self, enable=True, min_cells=1000000):
        """Overflow list: entries of >= min_cells cells are scored by bands on many warps (32-bit)."""
        self._check(self.lib.sw_set_overflow_wave(self.h, int(bool(enable)), int(min_cells)))

    def set_launch_plan(self, length_groups=2, query_groups=False):
        """length_groups: 0 one launch, 1 one launch per length group, 2 automatic; query_groups: variant per query length."""
        self._check(self.lib.sw_set_launch_plan(self.h, length_groups, int(bool(query_groups))))

    def set_pass_split(self, mode=-1):
        """Pass split of long queries: 0 never, -1 automatic, n >= 2 about n parts per work item."""
        self._check(self.lib.sw_set_pass_split(self.h, mode))

    @property
    def last_pass_parts(self):
        """Parts per work item of the last scoring call's plan (1 = not split)."""
        return int(self.lib.sw_last_pass_parts(self.h))

    def set_small_batch_path(self, enable):
        self._check(self.lib.sw_set_small_batch_path(self.h, int(bool(enable))))

    @property
    def device_error_bits(self):
        return int(self.lib.sw_device_error_bits(self.h))

    @property
    def batches_in_flight(self):
        return int(self.lib.sw_batches_in_flight(self.h))

    def fetch_ids(self):
        """ids of the batch fetched last (or of the resident database after load_db)."""
        ids = np.empty(self._ids_ns, dtype=np.uint64)
        self._check(self.lib.sw_fetch_ids(self.h, _ptr(ids), ids.size))
        return ids

    def score(self, queries, subjects, timeout_ms=-1):
        """Convenience: full score matrix [nq, ns]."""
        self.set_queries(queries)
        self.score_batch(subjects)
        return self.fetch(timeout_ms)

    # -- resident database ---------------------------------------------------------------
    def load_db(self, subjects, ids=None):
        packed, ln, off = self._as_packed(subjects)
        ids_a = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint64)
        self._check(self.lib.sw_load_db(self.h, _ptr(packed), _ptr(ln), _ptr(off), _ptr(ids_a), len(ln)))
        self.ns = len(ln)
        self._ids_ns = len(ln)
        self._db_len = ln.astype(np.uint64)

    def score_db(self):
        self._check(self.lib.sw_score_db(self.h))

    def wait(self, timeout_ms=-1):
        self._check(self.lib.sw_wait(self.h, timeout_ms))

    def fetch_db(self, out=None):
        i16 = self.out_mode == SW_OUTPUT_I16
        if out is None:
            out = np.empty((self.nq, self.ns), dtype=np.int16 if i16 else np.int32)
        fn = self.lib.sw_fetch_db_i16 if i16 else self.lib.sw_fetch_db
        self._check(fn(self.h, _ptr(out), out.size))
        return out

    def fetch_best(self):
        bs = np.empty(self.nq, dtype=np.int32)
        bi = np.empty(self.nq, dtype=np.uint64)
        self._check(self.lib.sw_fetch_best(self.h, _ptr(bs), _ptr(bi), self.nq))
        return bs, bi

    # -- introspection -------------------------------------------------------------------
    def set_kernel_choice(self, rows_per_lane=0, lanes_per_pair=0, force32=False, arith=-1):
        self._check(self.lib.sw_set_kernel_choice(self.h, rows_per_lane, lanes_per_pair, int(force32)))
        self._check(self.lib.sw_set_arith(self.h, arith))

    def set_autotune(self, enable):
        self._check(self.lib.sw_set_autotune(self.h, int(bool(enable))))

    def set_kernel_name(self, name):
        self._check(self.lib.sw_set_kernel_name(self.h, name.encode() if name else None))

    def stats(self):
        st = SwStats()
        self._check(self.lib.sw_get_stats(self.h, C.byref(st)))
        return {n: float(getattr(st, n)) for n, _ in SwStats._fields_}

    @property
    def last_kernel_ms(self):
        return float(self.lib.sw_last_kernel_ms(self.h))

    @property
    def kernel_launches(self):
        return int(self.lib.sw_kernel_launches(self.h))

    @property
    def last_cells(self):
        return int(self.lib.sw_last_cells(self.h))

    @property
    def last_kernel_name(self):
        return self.lib.sw_last_kernel_name(self.h).decode()


CIGAR_OPS = "MIDNSHP=X"      # BAM op codes 0 .. 8


def cigar_str(ops):
    """SAM text of BAM-encoded ops (len << 4 | op), e.g. "23=1I24="; "*" for no ops."""
    ops = np.asarray(ops, dtype=np.uint32).reshape(-1)
    if ops.size == 0:
        return "*"
    return "".join(f"{int(o) >> 4}{CIGAR_OPS[int(o) & 15]}" for o in ops)


def kernel_variants():
    L = load_library()
    return [L.sw_kernel_variant_name(i).decode() for i in range(L.sw_kernel_variant_count())]


def plan_pass_parts(npass, chunk_passes, chains, grid, mode=-1):
    """(split?, parts, passes per part) of the pass split for a launch of that shape (pure host arithmetic)."""
    n, pp = C.c_int(0), C.c_int(0)
    ok = load_library().sw_plan_pass_parts(npass, chunk_passes, chains, grid, mode, C.byref(n), C.byref(pp))
    return bool(ok), int(n.value), int(pp.value)


def plan_shards(lengths, n_shards):
    """Contiguous shard boundaries [n_shards + 1] as sw_load_db computes them (pure host)."""
    ln = np.ascontiguousarray(lengths, dtype=np.uint32)
    starts = np.zeros(n_shards + 1, dtype=np.uint64)
    rc = load_library().sw_plan_shards(_ptr(ln), len(ln), n_shards, _ptr(starts))
    if rc != SW_OK:
        raise SwError(rc, "sw_plan_shards")
    return starts


def set_fixed_penalty_kernels(enable):
    """False: never use the kernel instances with the default gap penalties compiled in."""
    load_library().sw_set_fixed_penalty_kernels(int(bool(enable)))


def params_in_exact_domain(match=5, mismatch=-4, gap_open=-12, gap_extend=-4, score_width=0):
    """1 = bit-exact vs the RTL for every input, 0 = accepted but the RTL is schedule-dependent
    there (SURVEY A.2), negative = rejected by sw_init."""
    p = SwParams(match, mismatch, gap_open, gap_extend, score_width)
    return int(load_library().sw_params_in_exact_domain(C.byref(p)))


def jit_compile_check(variant, gap_open, gap_extend):
    """(ok, message) of compiling / loading the run-time specialised instance of one variant."""
    buf = C.create_string_buffer(1024)
    rc = load_library().sw_jit_compile_check(variant.encode(), gap_open, gap_extend, buf, 1024)
    return rc, buf.value.decode(errors="replace")


def is_check_build():
    return bool(load_library().sw_is_check_build())


def device_count():
    return int(load_library().sw_device_count())
