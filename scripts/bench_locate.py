#!/usr/bin/env python3
"""Cost of locating hits (sw_locate_db) next to the scoring step that found them.  One JSON line, one GPU.

  python scripts/bench_locate.py [--subjects N] [--reps R] [--out path]

Config 3 (bench.py's workload: 10 M x 150 nt subjects resident, 1 % planted homologs, 100 x 150 nt queries) in hits
mode with a threshold that keeps the planted homologs:
  step    -- sw_score_db + sw_fetch_db_hits, host clock;
  locate  -- sw_locate_db on every hit, host clock around the blocking call, after one warm-up call;
  rates   -- located pairs per second, and cells per second of both passes (forward: qlen x slen of every pair;
             reverse: at most q_end x s_end, counted in full although the pass stops at the first cell reaching S);
  share   -- locate time over step time.
Two long-pair rows, where one thread per pair is the limit: 1 000 pairs of a 10 kb query x 1 kb subjects holding
mutated stretches of it, and one 20 kb x 20 kb pair (a mutated copy).  Checks inside the run: the located scores
equal the hit list's and, on the long rows, the int32 matrix's."""
import argparse
import importlib
import json
import os
import random
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("smith-waterman-fpga-module_b200")
import bench  # noqa: E402  (make_inputs: the same inputs bench.py scores)

MIN_SCORE = 200            # planted homologs of 150 nt score ~500-700; random pairs stay below ~60


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except OSError:
        return "nvidia-smi unavailable"


def cells(qlen, slen, co):
    """(forward, reverse) cells of the located pairs: qlen x slen, and q_end x s_end (an upper bound)."""
    fwd = int(np.sum(qlen.astype(np.uint64) * slen.astype(np.uint64)))
    rev = int(np.sum(co[:, 1].astype(np.uint64) * co[:, 3].astype(np.uint64)))
    return fwd, rev


def timed_locate(e, rows, idx, reps):
    e.locate_db(rows, idx)                            # warm-up: module load, scratch and staging allocation
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        sc, co = e.locate_db(rows, idx)
        times.append(time.perf_counter() - t0)
    return statistics.median(times), times, sc, co


def row_record(name, n, t, times, fwd, rev):
    return {"case": name, "pairs": n, "locate_s_median": t, "locate_s": [round(x, 5) for x in times],
            "pairs_per_s": n / t, "cells_forward": fwd, "cells_reverse_max": rev, "gcups_both_passes": (fwd + rev) / t / 1e9}


def config3(ns, reps):
    q, db = bench.make_inputs(pkg, ns, 100, 0)
    with pkg.Engine() as e:
        e.set_queries(q)
        e.load_db(db)
        e.set_hits(MIN_SCORE)
        e.score_db()                                  # warm-up: autotune, allocations
        e.fetch_db_hits()
        steps = []
        for _ in range(reps):
            t0 = time.perf_counter()
            e.score_db()
            row, idx, hsc = e.fetch_db_hits()
            steps.append(time.perf_counter() - t0)
        kernel = e.last_kernel_name
        t, times, sc, co = timed_locate(e, row, idx, reps)
        assert e.device_error_bits == 0
    assert np.array_equal(sc, hsc), "located scores differ from the hit list"
    fwd, rev = cells(q[1][row], db[1][idx], co)
    step = statistics.median(steps)
    rec = row_record(f"config 3: {ns} x 150 nt (1 % planted homologs) vs 100 x 150 nt, hits >= {MIN_SCORE}",
                     len(row), t, times, fwd, rev)
    rec.update({"step_s_median": step, "step_s": [round(x, 4) for x in steps], "step_kernel": kernel,
                "locate_share_of_step": t / step})
    return rec


def long_pairs(name, query, subjects, reps):
    with pkg.Engine() as e:
        e.set_queries([query])
        e.load_db(subjects)
        e.score_db()
        mat = e.fetch_db()
        rows = np.zeros(len(subjects), np.uint32)
        idx = np.arange(len(subjects), dtype=np.uint64)
        t, times, sc, co = timed_locate(e, rows, idx, reps)
        assert e.device_error_bits == 0
    assert np.array_equal(sc, mat[0]), "located scores differ from the int32 matrix"
    fwd, rev = cells(np.full(len(subjects), len(query)), np.array([len(s) for s in subjects]), co)
    rec = row_record(name, len(subjects), t, times, fwd, rev)
    rec["score_max"] = int(sc.max())
    return rec


def mutate(rng, s, psub, pindel):
    out = []
    for ch in s:
        r = rng.random()
        if r < pindel / 2:
            continue
        if r < pindel:
            out.append(rng.choice("ACGT"))
        out.append(rng.choice("ACGT") if rng.random() < psub else ch)
    return "".join(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subjects", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON record to this file")
    a = ap.parse_args()
    rng = random.Random(2026)
    rand = lambda n: "".join(rng.choice("ACGT") for _ in range(n))  # noqa: E731
    q10k = rand(10_000)
    subs1k = []
    for _ in range(1000):
        p = rng.randrange(0, 10_000 - 600)
        core = mutate(rng, q10k[p:p + rng.randint(100, 600)], 0.05, 0.02)
        subs1k.append((rand(rng.randint(0, 400)) + core + rand(1000))[:1000])
    q20k = rand(20_000)
    rec = {"gpu": gpu_info(),
           "config3": config3(a.subjects, a.reps),
           "long_10kb_x_1kb": long_pairs("1 000 pairs: 10 kb query x 1 kb subjects", q10k, subs1k, a.reps),
           "long_20kb_x_20kb": long_pairs("1 pair: 20 kb x 20 kb (mutated copy)", q20k,
                                          [mutate(rng, q20k, 0.05, 0.02)[:20_000]], 1)}
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
