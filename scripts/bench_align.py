#!/usr/bin/env python3
"""Cost of aligning hits (sw_align_db: locate, then one traceback pass over each located rectangle) next to locating
them (sw_locate_db) and the scoring step that found them.  One JSON line, one GPU.

  python scripts/bench_align.py [--subjects N] [--reps R] [--out path]

Config 3 (bench.py's workload: 10 M x 150 nt subjects resident, 1 % planted homologs, 100 x 150 nt queries) in hits
mode at T = 200, which keeps the planted homologs:
  step    -- sw_score_db + sw_fetch_db_hits, host clock;
  locate  -- sw_locate_db on every hit, host clock around the blocking call, after one warm-up call;
  align   -- sw_align_db on the same hits, the same way;
  cells   -- rectangle cells of the traceback pass ((q_end - q_begin) x (s_end - s_begin) of every pair).
One long-pair row, where one thread per pair is the limit: 1 000 pairs of a 10 kb query x 1 kb subjects holding
mutated stretches of it.  Checks inside the run: the aligned scores and coordinates equal sw_locate_db's, and the
ops of every pair score its score under the combined-gap rule."""
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
MATCH, MISMATCH, GAP_OPEN, GAP_EXTEND = 5, -4, -12, -4      # the Engine's defaults


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except OSError:
        return "nvidia-smi unavailable"


def timed(fn, reps):
    fn()                                              # warm-up: module load, scratch and staging allocation
    times, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), times, out


def op_scores(off, cig):
    """Each pair's score from its ops: a maximal run of I / D columns costs gap_open + gap_extend * length."""
    ln = (cig >> 4).astype(np.int64)
    op = cig & 15
    per = np.where(op == 7, MATCH * ln, np.where(op == 8, MISMATCH * ln, GAP_EXTEND * ln))
    gap = (op == 1) | (op == 2)
    prev_gap = np.concatenate([[False], gap[:-1]])
    starts = np.zeros(len(cig), bool)
    starts[off[:-1][off[:-1] < off[1:]].astype(np.int64)] = True
    per += np.where(gap & (~prev_gap | starts), GAP_OPEN, 0)     # a gap run opens here
    total = np.concatenate([[0], np.cumsum(per)])
    return total[off[1:].astype(np.int64)] - total[off[:-1].astype(np.int64)]


def measure(e, rows, idx, reps):
    t_loc, loc_times, (lsc, lco) = timed(lambda: e.locate_db(rows, idx), reps)
    t_aln, aln_times, (sc, co, off, cig) = timed(lambda: e.align_db(rows, idx), reps)
    assert e.device_error_bits == 0
    assert np.array_equal(sc, lsc) and np.array_equal(co, lco), "aligned scores / coordinates differ from locate's"
    assert np.array_equal(op_scores(off, cig), sc.astype(np.int64)), "ops do not score the located score"
    rect = int(np.sum((co[:, 1] - co[:, 0]).astype(np.uint64) * (co[:, 3] - co[:, 2]).astype(np.uint64)))
    return {"pairs": len(rows), "locate_s_median": t_loc, "locate_s": [round(x, 5) for x in loc_times],
            "align_s_median": t_aln, "align_s": [round(x, 5) for x in aln_times],
            "align_over_locate": t_aln / t_loc, "rectangle_cells": rect, "ops": int(len(cig)),
            "pairs_per_s_align": len(rows) / t_aln}


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
        rec = measure(e, row, idx, reps)
    step = statistics.median(steps)
    rec.update({"case": f"config 3: {ns} x 150 nt (1 % planted homologs) vs 100 x 150 nt, hits >= {MIN_SCORE}",
                "step_s_median": step, "step_s": [round(x, 4) for x in steps], "step_kernel": kernel,
                "locate_share_of_step": rec["locate_s_median"] / step, "align_share_of_step": rec["align_s_median"] / step})
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


def long_pairs(query, subjects, reps):
    with pkg.Engine() as e:
        e.set_queries([query])
        e.load_db(subjects)
        e.score_db()
        e.wait()
        rec = measure(e, np.zeros(len(subjects), np.uint32), np.arange(len(subjects), dtype=np.uint64), reps)
    rec["case"] = "1 000 pairs: 10 kb query x 1 kb subjects"
    return rec


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
    rec = {"gpu": gpu_info(),
           "config3": config3(a.subjects, a.reps),
           "long_10kb_x_1kb": long_pairs(q10k, subs1k, a.reps)}
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
