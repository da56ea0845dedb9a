#!/usr/bin/env python3
"""Hit-list output against the int16 matrix on config 3 (bench.py's workload: 10 M x 150 nt subjects, 1 %
planted homologs, 100 x 150 nt queries), one GPU, the bench kernel forced in both arms.  One JSON line.

  python scripts/bench_hits.py [n_subjects] [reps]

Arms, alternated within the process (host buffers pinned, as in bench.py's end-to-end arm):
  (a) int16 matrix: sw_score_batch + sw_fetch_i16 (2 GB of D2H per step at full size);
  (b) hit list:     sw_score_batch + sw_fetch_hits with T above the random-pair maximum.
Both report end-to-end seconds per step, kernel time (CUDA events), D2H bytes and the fetch phase times of
sw_get_stats.  Checks inside the run: (1) the hits of 4 queries equal their GPU int32 matrix filtered at T;
(2) one query's hits over a 20 000-subject sample equal the CPU oracle's scores filtered at T."""
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
T = 100                    # random 150 x 150 pairs score far below (the sample's maximum is reported)
KERNEL = "strip_s16x2_R25x2_G1_U4_F31"
SAMPLE = 20000


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


q, db = bench.make_inputs(pkg, NS, NQ, 0)
hdb = tuple(pinned(x) for x in db)
import torch  # noqa: E402
out16 = torch.empty((NQ, NS), dtype=torch.int16, pin_memory=True).numpy()

arms = {"int16_matrix": [], "hits": []}
with pkg.Engine() as e:
    e.set_kernel_name(KERNEL)
    e.set_queries(q)

    def run(arm):
        if arm == "int16_matrix":
            e.set_hits(0)
            e.set_output(pkg.SW_OUTPUT_I16)
        else:
            e.set_hits(T, 1 << 22)
        t0 = time.perf_counter()
        e.score_batch(hdb)
        if arm == "int16_matrix":
            e.fetch(out=out16)
            res, d2h = None, out16.nbytes
        else:
            res = e.fetch_hits()
            d2h = res[0].size * 12 + 4
        wall = time.perf_counter() - t0
        st = e.stats()
        return {"e2e_s": wall, "kernel_ms": e.last_kernel_ms, "d2h_bytes": d2h, "fetch_wait_ms": st["fetch_wait_ms"],
                "fetch_drain_ms": st["fetch_drain_ms"], "kernel": e.last_kernel_name}, res

    for arm in arms:                                   # warm-up of both shapes (module load, allocations, sort)
        run(arm)
    hits = None
    for _ in range(REPS):
        for arm in arms:
            rec, res = run(arm)
            arms[arm].append(rec)
            if res is not None:
                hits = res
    cells = e.last_cells
    # (1) four queries in int32 matrix mode on the GPU, filtered at T on the host
    pick = [0, 1, NQ // 2, NQ - 1]
    nb = 38
    sub_q = (np.concatenate([q[0][int(q[2][i]): int(q[2][i]) + nb] for i in pick] + [np.zeros(16, np.uint8)]),
             q[1][pick], (np.arange(len(pick), dtype=np.uint64) * nb))
    e.set_hits(0)
    e.set_output(pkg.SW_OUTPUT_I32)
    e.set_kernel_name("")
    e.set_queries(sub_q)
    e.load_db(db)
    e.score_db()
    mat = e.fetch_db()

row, idx, sc = hits
for k, qi in enumerate(pick):
    sel = row == qi
    want_i = np.nonzero(mat[k] >= T)[0]
    assert np.array_equal(idx[sel], want_i.astype(np.uint64)) and np.array_equal(sc[sel], mat[k, want_i]), \
        f"hits of query {qi} differ from its GPU int32 matrix filtered at T"
# (2) query 0 against the first SAMPLE subjects on the CPU oracle
from oracle import oracle as om  # noqa: E402
om.build_oracle()
o = om.Oracle()
nbs = int(db[2][SAMPLE]) if SAMPLE < NS else db[0].size
cpu, used = o.score_batch_packed(sub_q[0], sub_q[1][:1], sub_q[2][:1], db[0][:nbs + 16], db[1][:SAMPLE], db[2][:SAMPLE])
sel = (row == 0) & (idx < SAMPLE)
want_i = np.nonzero(cpu[0] >= T)[0]
assert np.array_equal(idx[sel], want_i.astype(np.uint64)) and np.array_equal(sc[sel], cpu[0, want_i]), \
    "hits of query 0 differ from the CPU oracle filtered at T"
planted = np.zeros(SAMPLE, bool)
planted[::100] = True                              # plant_homologs(frac=0.01): every 100th subject
random_max = int(cpu[0, ~planted].max())


def summary(recs):
    med = lambda k: statistics.median(r[k] for r in recs)  # noqa: E731
    return {"e2e_s_median": med("e2e_s"), "e2e_s": [round(r["e2e_s"], 4) for r in recs],
            "kernel_ms_median": med("kernel_ms"), "e2e_gcups": cells / med("e2e_s") / 1e9,
            "kernel_gcups": cells / med("kernel_ms") / 1e6, "d2h_bytes": recs[-1]["d2h_bytes"],
            "fetch_wait_ms_median": med("fetch_wait_ms"), "fetch_drain_ms_median": med("fetch_drain_ms"),
            "kernel": recs[-1]["kernel"]}


print(json.dumps({"workload": f"config 3: {NS} x 150 nt subjects (1 % planted homologs) vs {NQ} x 150 nt queries, 1 GPU, "
                              f"streaming (sw_score_batch + fetch), kernel {KERNEL} forced in both arms",
                  "gpu": gpu_info(), "min_score": T, "hits": int(row.size), "reps": REPS,
                  "int16_matrix": summary(arms["int16_matrix"]), "hits_list": summary(arms["hits"]),
                  "checked": f"{len(pick)} queries vs their GPU int32 matrix filtered at T; query 0 vs the CPU oracle on "
                             f"{SAMPLE} subjects ({used} threads)",
                  "random_pair_max_in_sample": random_max}))
