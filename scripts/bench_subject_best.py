#!/usr/bin/env python3
"""Per-subject best output against the int16 matrix on config 3 (bench.py's workload: 10 M x 150 nt subjects, 1 %
planted homologs, 100 x 150 nt queries), one GPU, the bench kernel forced in both arms.  One JSON line.

  python scripts/bench_subject_best.py [n_subjects] [reps]

Arms, alternated within the process (host buffers pinned, as in bench.py's end-to-end arm):
  (a) int16 matrix:   sw_score_batch + sw_fetch_i16 (2 GB of D2H per step at full size);
  (b) subject best:   sw_score_batch + sw_fetch_subject_best (12 bytes per subject: 120 MB at full size).
Both report end-to-end seconds per step, kernel time (CUDA events), D2H bytes and the fetch phase times of
sw_get_stats.  Checks inside the run: (1) the result over the first 200 000 subjects equals the column maximum,
argmax and runner-up of the same handle's int32 matrix; (2) the first 2 000 subjects equal the CPU oracle's."""
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("smith-waterman-fpga-module_b200")
import bench  # noqa: E402  (make_inputs: the same inputs bench.py scores)

NS = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
NQ = 100
KERNEL = "strip_s16x2_R25x2_G1_U4_F31"
SLICE = min(200_000, NS)   # check (1): subjects compared with the GPU int32 matrix
SAMPLE = min(2000, NS)     # check (2): subjects compared with the CPU oracle


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except OSError:
        return "nvidia-smi unavailable"


def pinned(a):
    import torch
    return torch.from_numpy(a).pin_memory().numpy()


def expected(mat):
    """(best score, lowest best row, runner-up score) of every column of an int32 matrix."""
    return mat.max(0), mat.argmax(0).astype(np.uint32), np.sort(mat, 0)[-2]


def head(db, n):
    """The first n subjects of a packed database (same packed buffer, shorter length / offset arrays)."""
    nbytes = int(db[2][n]) if n < db[1].size else db[0].size
    return db[0][:nbytes + 16], db[1][:n], db[2][:n]


q, db = bench.make_inputs(pkg, NS, NQ, 0)
hdb = tuple(pinned(x) for x in db)
import torch  # noqa: E402
out16 = torch.empty((NQ, NS), dtype=torch.int16, pin_memory=True).numpy()

arms = {"int16_matrix": [], "subject_best": []}
with pkg.Engine() as e:
    e.set_kernel_name(KERNEL)
    e.set_queries(q)

    def run(arm):
        e.set_subject_best(arm == "subject_best")
        if arm == "int16_matrix":
            e.set_output(pkg.SW_OUTPUT_I16)
        t0 = time.perf_counter()
        e.score_batch(hdb)
        if arm == "int16_matrix":
            e.fetch(out=out16)
            res, d2h = None, out16.nbytes
        else:
            res = e.fetch_subject_best()
            d2h = NS * 12
        wall = time.perf_counter() - t0
        st = e.stats()
        return {"e2e_s": wall, "kernel_ms": e.last_kernel_ms, "d2h_bytes": d2h, "fetch_wait_ms": st["fetch_wait_ms"],
                "fetch_drain_ms": st["fetch_drain_ms"], "kernel": e.last_kernel_name}, res

    for arm in arms:                                   # warm-up of both shapes (module load, allocations)
        run(arm)
    best = None
    for _ in range(REPS):
        for arm in arms:
            rec, res = run(arm)
            arms[arm].append(rec)
            if res is not None:
                best = res
    cells = e.last_cells
    # (1) the first SLICE subjects in int32 matrix mode on the same handle
    e.set_subject_best(False)
    e.set_output(pkg.SW_OUTPUT_I32)
    e.score_batch(head(db, SLICE))
    mat = e.fetch()

for name, g, w in zip(("best_score", "best_row", "second_score"), best, expected(mat)):
    assert np.array_equal(g[:SLICE], w), f"{name} differs from the same handle's int32 matrix on {SLICE} subjects"
# (2) all queries against the first SAMPLE subjects on the CPU oracle
from oracle import oracle as om  # noqa: E402
om.build_oracle()
o = om.Oracle()
cpu, used = o.score_batch_packed(q[0], q[1], q[2], *head(db, SAMPLE))
for name, g, w in zip(("best_score", "best_row", "second_score"), best, expected(cpu)):
    assert np.array_equal(g[:SAMPLE], w), f"{name} differs from the CPU oracle on {SAMPLE} subjects"


def summary(recs):
    med = lambda k: statistics.median(r[k] for r in recs)  # noqa: E731
    return {"e2e_s_median": med("e2e_s"), "e2e_s": [round(r["e2e_s"], 4) for r in recs],
            "kernel_ms_median": med("kernel_ms"), "e2e_gcups": cells / med("e2e_s") / 1e9,
            "kernel_gcups": cells / med("kernel_ms") / 1e6, "d2h_bytes": recs[-1]["d2h_bytes"],
            "fetch_wait_ms_median": med("fetch_wait_ms"), "fetch_drain_ms_median": med("fetch_drain_ms"),
            "kernel": recs[-1]["kernel"]}


print(json.dumps({"workload": f"config 3: {NS} x 150 nt subjects (1 % planted homologs) vs {NQ} x 150 nt queries, 1 GPU, "
                              f"streaming (sw_score_batch + fetch), kernel {KERNEL} forced in both arms",
                  "gpu": gpu_info(), "reps": REPS,
                  "int16_matrix": summary(arms["int16_matrix"]), "subject_best": summary(arms["subject_best"]),
                  "subjects_with_a_margin": int((best[0] > best[2]).sum()),
                  "checked": f"{SLICE} subjects vs the same handle's int32 matrix; {SAMPLE} subjects x {NQ} queries vs the "
                             f"CPU oracle ({used} threads)"}))
