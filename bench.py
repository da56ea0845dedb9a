#!/usr/bin/env python3
"""bench.py -- GCUPS of the score-only Smith-Waterman hot path on B200.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on):
synthetic iid-uniform 150-nt subjects (10 M per GPU, weak scaling) against 100 x 150-nt
queries, penalties 5/-4/-12/-4, inter-task strip kernel.  One "step" = one pass of the
hot path over the whole resident database shard for all queries.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm
  python bench.py --impl reference [...]                         CPU arm (oracle port, all host threads)
  torchrun --nproc-per-node N bench.py --gpus N ...              one rank per GPU, no collective on the data path
  python bench.py ... --dump-outputs DIR                         also write the last timed step's scores to DIR/*.npy

Prints ONE JSON line (rank 0).  `value` = device-resident kernel throughput (CUDA events on
the launching stream, max over ranks); `e2e` = the same metric through sw_score_batch /
sw_fetch with pinned HOST buffers, H2D + D2H inside the timed region.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

QLEN = 150
TLEN = 150
SEED = 20160912
SM_COUNT = 148
PIPE_PROFILE = "profiles/r01_pipe_pairs_1024thr.json"
SASS_PROFILE = "profiles/r02_sass_hotloop.json"
DUMP_BYTES = 60_000_000


def measured_r_int():
    """Issue rate of the packed 16-bit DPX / min-max instructions (thread-instr / clk / SM), as
    MEASURED by microbench/pipe_pairs.cu on this pool's B200 and committed under profiles/."""
    with open(os.path.join(ROOT, PIPE_PROFILE)) as f:
        rows = json.load(f)["results"]
    alone = [r["thread_instr_per_clk_per_sm"] for r in rows
             if r["nb"] == 0 and r["a"] in ("VIADDMNMX.S16x2", "VIMNMX.S16x2", "VIMNMX3.S16x2")]
    return min(alone)


def alu_instr_per_cell_pair(kname):
    """ALU-pipe instructions per two cells in the hot loop of the bench kernel, counted from its SASS
    (scripts/sass_hotloop.py -> profiles/r02_sass_hotloop.json); 3.5 by construction (DESIGN.md 2)."""
    try:
        with open(os.path.join(ROOT, SASS_PROFILE)) as f:
            d = json.load(f)
        k = d["kernels"].get(kname)
        if k:
            return float(k["alu_pipe_per_cell_pair"]), float(k["issue_slots_per_cell_pair"]), SASS_PROFILE
    except Exception:
        pass
    return 3.5, None, "DESIGN.md section 2 (no SASS histogram for this kernel)"


def peaks():
    p = {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p = {"hbm_gbs": float(m["hbm_gbs"]), "sm_max_mhz": float(m["sm_max_mhz"]), "source": "measured"}
    except Exception:
        pass
    return p


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU with nvidia-smi while a region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 7:
                self.rows.append(f)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for f in self.rows:
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """All cores this process may use (torchrun sets OMP_NUM_THREADS=1; the CPU arm must not inherit that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def make_inputs(pkg, n_subjects, n_queries, rank):
    db = pkg.random_packed_db(n_subjects, TLEN, seed=SEED + 1000 * rank)
    q = pkg.random_packed_db(n_queries, QLEN, seed=SEED - 1)
    # 1 % of the subjects are homologs of a query (5 % substitutions, 2 % indels) so that the gap
    # path carries real alignments (SURVEY section 8d, config 3); the kernel has no data-dependent exit
    pkg.plant_homologs(db, q, 0.01, seed=SEED + 7 + rank)
    return q, db


def base_config(args):
    """Identical for both arms (the driver compares the two `config` objects)."""
    return {"workload": workload_name(args), "queries": args.queries, "query_len": QLEN, "subject_len": TLEN,
            "subjects_per_gpu": args.subjects, "penalties": "5/-4/-12/-4",
            "planted_homologs": "1 % of subjects = a query with 5 % substitutions + 2 % indels",
            "l2": "inputs (code stream + score matrix per GPU) larger than L2"}


def run_reference(args, rank, world):
    """CPU arm: the oracle port of the PE recurrence (the reference ships no CPU scorer and its
    RTL cannot be simulated here, DESIGN.md), all host threads, bounded sample per step."""
    if rank != 0:
        return
    from oracle import oracle as om
    om.build_oracle()
    o = om.Oracle()
    pkg_seq = importlib.import_module("smith-waterman-fpga-module_b200.seqio")
    ns = args.ref_subjects
    q = pkg_seq.random_packed_db(args.queries, QLEN, seed=SEED - 1)
    db = pkg_seq.random_packed_db(ns, TLEN, seed=SEED)
    pkg_seq.plant_homologs(db, q, 0.01, seed=SEED + 7)
    cells = ns * TLEN * args.queries * QLEN
    used = 1
    for _ in range(max(args.warmup, 0)):
        _, used = o.score_batch_packed(q[0], q[1], q[2], db[0][: (ns // 8) * 38 + 16], db[1][: ns // 8], db[2][: ns // 8],
                                       nthreads=host_threads())
    t0 = time.perf_counter()
    for _ in range(args.steps):
        scores, used = o.score_batch_packed(q[0], q[1], q[2], db[0], db[1], db[2], nthreads=host_threads())
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, scores)
    gcups = cells * args.steps / dt / 1e9
    sample = (f"each step scores the first {ns} of the {args.subjects} synthetic 150-nt subjects x {args.queries} "
              f"queries ({cells:.3g} cells); GCUPS is a rate, so the bounded sample does not change the metric")
    line = {"impl": "reference", "metric": "GCUPS (score-only SW)", "value": gcups, "unit": "GCUPS",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic", "config": base_config(args),
            "cpu_baseline": {"value": gcups, "unit": "GCUPS", "cores": used, "kind": "port", "sample": sample,
                             "note": "scalar, un-vectorised int32 C port of the PE recurrence (the reference has no CPU "
                                     "scorer): context for the GPU number, not a tuned CPU competitor"},
            "e2e": {"value": gcups, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_name(args):
    return (f"configs[2]: synthetic {args.subjects} x {TLEN} nt subjects per GPU vs {args.queries} x {QLEN} nt "
            f"queries, inter-task kernel")


_REAL_STDOUT = None


def capture_stdout():
    """stdout must carry exactly ONE JSON line, but libraries print there too (NCCL's version banner
    at communicator creation).  Point fd 1 at stderr for the whole run and keep the real stdout for
    the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def matrices_equal(a, b):
    """Row-wise comparison of two score matrices of possibly different integer width."""
    return a.shape == b.shape and all(np.array_equal(a[i], b[i]) for i in range(a.shape[0]))


def dump_outputs(path, scores):
    """Writes the [queries, subjects] score matrix the timed path returned as float32, which holds every
    score exactly.  A matrix above DUMP_BYTES (the default GPU workload's is 4 GB) is cut to a fixed-seed
    sample of its columns, sorted; subject_index.npy names the columns kept.  Two builds run with the
    same arguments score the same inputs, so their files compare element for element."""
    nq, ns = scores.shape
    ncol = min(ns, DUMP_BYTES // (4 * nq + 8))
    idx = np.sort(np.random.default_rng(SEED).choice(ns, size=ncol, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "scores.npy"), scores[:, idx].astype(np.float32))
    np.save(os.path.join(path, "subject_index.npy"), idx.astype(np.float64))
    log(f"wrote scores of {ncol} of {ns} subjects x {nq} queries to {path}")


def e2e_loop(eng, hdb, out, steps):
    """Streaming use of the ABI: step k+1 is submitted (sort, H2D, kernels enqueued) before the scores
    of step k are fetched -- two batches in flight, every byte still crosses PCIe each step."""
    t0 = time.perf_counter()
    eng.score_batch(hdb)
    for k in range(steps):
        if k + 1 < steps:
            eng.score_batch(hdb)
        eng.fetch(out=out)
    return time.perf_counter() - t0


def single_handle_phase(pkg, torch, args, world, q, hdb, out, chk, e2e_1gpu_s):
    """north_star partition (SURVEY 8e): ONE handle, ONE database sharded over all N GPUs of the box,
    host-side gather into the caller's [nq][ns] matrix (ScoreBank_v2.v:78-139,162 at the GPU level).
    Strong scaling of the literal config 3: the same 10 M x 150 database, 1 GPU vs N GPUs, end to end
    with host buffers.  Runs on rank 0 while the other ranks idle on a CPU (gloo) barrier."""
    steps = max(2, args.e2e_steps)
    res = {"n_gpus": world, "subjects_total": int(len(hdb[1])), "steps": steps,
           "api": "sw_init(gpu_ids=0..N-1) + sw_score_batch + sw_fetch_i16, pinned host buffers, two batches in flight"}
    # 1 GPU, alone on the box (the per-rank e2e above ran with N ranks sharing the host)
    if world > 1:
        with pkg.Engine(gpu_ids=[0]) as e1:
            e1.set_output(pkg.SW_OUTPUT_I16)
            e1.set_queries(q)
            e1.score_batch(hdb); e1.fetch(out=out)
            t1 = e2e_loop(e1, hdb, out, steps) / steps
            cells = e1.last_cells
            res["kernel_1gpu"] = e1.last_kernel_name
    else:
        t1 = e2e_1gpu_s
        cells = None
    with pkg.Engine(gpu_ids=list(range(world))) as en:
        en.set_output(pkg.SW_OUTPUT_I16)
        en.set_queries(q)
        en.score_batch(hdb); en.fetch(out=out)            # warm-up (autotune, allocations)
        tn = e2e_loop(en, hdb, out, steps) / steps
        cells = en.last_cells
        res["kernel_ms_max_over_gpus"] = en.last_kernel_ms
        res["kernel"] = en.last_kernel_name
        st = en.stats() if hasattr(en, "stats") else None
        if st:
            res["host_ms"] = st
    equal = bool(matrices_equal(out, chk))
    assert equal, "single-handle N-GPU score matrix differs from the 1-GPU result"
    res.update({"value": cells / tn / 1e9, "unit": "GCUPS", "ms_per_step": tn * 1e3,
                "value_1gpu": cells / t1 / 1e9, "ms_per_step_1gpu": t1 * 1e3,
                "strong_eff": (t1 / tn) / world, "matrix_equal_to_1gpu": equal,
                "d2h_bytes_per_step": int(out.nbytes), "h2d_bytes_per_step": int(sum(a.nbytes for a in hdb))})
    # what bounds it: device time vs host-visible step time
    res["device_bound_frac"] = res["kernel_ms_max_over_gpus"] / (tn * 1e3)
    return res


def main():
    capture_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--subjects", type=int, default=10_000_000, help="subjects per GPU")
    ap.add_argument("--queries", type=int, default=100)
    ap.add_argument("--ref-subjects", type=int, default=4000, help="subjects per step of the CPU arm")
    ap.add_argument("--cpu-subjects", type=int, default=20000, help="subjects of the cpu_baseline sample")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--rows", type=int, default=0, help="force rows-per-lane of the strip kernel")
    ap.add_argument("--lanes", type=int, default=0, help="force lanes-per-pair of the strip kernel")
    ap.add_argument("--arith", type=int, default=-1, help="-1 auto, 0 s16x2")
    ap.add_argument("--kernel", default="", help="force a strip-kernel variant by name")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-single-handle", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs{} / latency{} blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the score matrix of the last one (rank 0's shard; a "
                         "fixed-seed sample of its columns) to DIR/scores.npy + DIR/subject_index.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        emit({"error": "no CUDA device: this bench has no CPU fallback"})
        return 1
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's version banner off it
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")     # host-side barrier: waiting ranks keep their GPU idle

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    pkg = importlib.import_module("smith-waterman-fpga-module_b200")
    q, db = make_inputs(pkg, args.subjects, args.queries, rank)
    eng = pkg.Engine(gpu_ids=[local_rank])
    eng.set_kernel_choice(args.rows, args.lanes, False, args.arith)
    if args.kernel:
        eng.set_kernel_name(args.kernel)
    eng.set_queries(q)

    # ---- device-resident arm: database uploaded once, then K timed passes -------------------
    eng.load_db(db)
    for _ in range(args.warmup):
        eng.score_db()
        eng.wait()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches
    kernel_ms = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.score_db()
        eng.wait()
        kernel_ms.append(eng.last_kernel_ms)        # CUDA events on the library's compute stream
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.kernel_launches - launches0
    cells_step = eng.last_cells
    kname = eng.last_kernel_name
    dev_s = max_over_ranks(sum(kernel_ms) / 1e3)
    wall_s = max_over_ranks(wall)
    gcups = cells_step * world * args.steps / dev_s / 1e9
    log(f"resident arm: {gcups:.1f} GCUPS, kernel {kname}")
    # spot check: the timed output is the real thing (compare a slice with an independent launch)
    chk = eng.fetch_db()
    checksum = int(chk[:, :: max(1, args.subjects // 4096)].astype(np.int64).sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, chk)

    # ---- end-to-end arm: host buffers in, host scores out, every step -----------------------
    e2e = None
    hdb = out = None
    e2e_s_local = None
    if not args.no_e2e:
        pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
        hdb = (pin(db[0]), pin(db[1]), pin(db[2]))
        # the score matrix is fetched as int16 (scores <= 5 x 150 fit; anything above 32767 would come
        # back through the overflow side list): half the D2H bytes of the int32 matrix
        eng.set_output(pkg.SW_OUTPUT_I16)
        out = torch.empty((args.queries, args.subjects), dtype=torch.int16, pin_memory=True).numpy()
        eng.score_batch(hdb); eng.fetch(out=out)          # warm-up
        barrier()
        e2e_s_local = e2e_loop(eng, hdb, out, args.e2e_steps)
        barrier()
        e2e_s = max_over_ranks(e2e_s_local)
        assert matrices_equal(out, chk), "e2e scores differ from the resident-path scores"
        assert eng.fetch_overflow()[0].size == 0
        e2e = {"value": cells_step * world * args.e2e_steps / e2e_s / 1e9, "unit": "GCUPS",
               "h2d_bytes_per_step": int(sum(a.nbytes for a in hdb)) * world, "d2h_bytes_per_step": int(out.nbytes) * world,
               "ms_per_step": e2e_s / args.e2e_steps * 1e3, "steps": args.e2e_steps,
               "api": "sw_score_batch + sw_fetch_i16 (two batches in flight), pinned host buffers, int16 score matrix"}
        log(f"e2e arm: {e2e['value']:.1f} GCUPS")

    # ---- CPU baseline (rank 0, N=1 only): the oracle port on a bounded sample ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import oracle as om
        om.build_oracle()
        o = om.Oracle()
        ns = min(args.cpu_subjects, args.subjects)
        nb = (TLEN + 3) // 4
        t0 = time.perf_counter()
        ref, used = o.score_batch_packed(q[0], q[1], q[2], db[0][: ns * nb + 16], db[1][:ns], db[2][:ns],
                                         nthreads=host_threads())
        dt = time.perf_counter() - t0
        assert np.array_equal(ref, chk[:, :ns]), "GPU scores differ from the CPU oracle on the sample"
        cpu = {"value": ns * TLEN * args.queries * QLEN / dt / 1e9, "unit": "GCUPS", "cores": used, "kind": "port",
               "sample": f"first {ns} subjects x {args.queries} queries ({ns * TLEN * args.queries * QLEN:.3g} cells), "
                         f"scalar int32 C oracle, OpenMP; scores equal to the GPU's"}

    # ---- configs 2 / 4 / 5 and the latency regime (rank 0, N=1): driver-visible evidence -----
    extra = {}
    if rank == 0 and world == 1 and not args.no_configs:
        try:
            from scripts import bench_configs as bc
            eng.close()
            extra = bc.bench_blocks(pkg, log)
        except Exception as ex:           # the headline line must still be printed
            extra = {"configs_error": repr(ex)}

    # ---- single handle over all GPUs (strong scaling of the literal config 3) ----------------
    single = None
    if not args.no_e2e and not args.no_single_handle and world > 1:
        eng.close()
        torch.cuda.empty_cache()
        barrier()
        if rank == 0:
            try:
                single = single_handle_phase(pkg, torch, args, world, q, hdb, out, chk, e2e_s_local / args.e2e_steps)
                log(f"single handle over {world} GPUs: {single['value']:.1f} GCUPS, strong_eff {single['strong_eff']:.3f}")
            except Exception as ex:
                single = {"error": repr(ex)}
        dist.barrier(group=cpu_group)
    elif not args.no_e2e and world == 1 and e2e is not None:
        single = {"n_gpus": 1, "value": e2e["value"], "unit": "GCUPS", "ms_per_step": e2e["ms_per_step"],
                  "strong_eff": 1.0, "note": "N = 1: the e2e arm is the single-handle path"}

    if rank == 0:
        pk = peaks()
        r_int = measured_r_int()
        per_gpu = gcups / world
        arith = "s16x2" if "s16x2" in kname else "int32"
        # ALU-pipe instructions per cell pair of the chosen kernel, counted in its SASS; the adds of the
        # recurrence run on the FMA-side pipe and co-issue (profiles/r01_pipe_pairs_1024thr.json)
        if arith == "s16x2":
            alu_per_pair, issue_per_pair, alu_src = alu_instr_per_cell_pair(kname)
        else:
            alu_per_pair, issue_per_pair, alu_src = 12.0, None, "32-bit fallback"
        pipe_gcups = SM_COUNT * pk["sm_max_mhz"] * 1e6 * r_int * 2.0 / alu_per_pair / 1e9
        survey_gcups = SM_COUNT * pk["sm_max_mhz"] * 1e6 * r_int * 2.0 / 6.0 / 1e9
        # per launch: the pair's code stream (one byte per column) + pair_len + pair_subj, read once;
        # plus one int32 score per (query, subject) written once
        n_launch = max(1, launches // max(1, args.steps))
        algo_bytes = (args.subjects / 2) * (((TLEN + 3) // 4) * 4 + 8 + 8) * n_launch + args.subjects * args.queries * 4
        traffic = None
        for tf in ("r02_traffic.json", "r01_traffic.json"):
            try:
                with open(os.path.join(ROOT, "profiles", tf)) as f:
                    tr = json.load(f)
                if tr["kernel"] == kname and tr["subjects_per_gpu"] == args.subjects and tr["queries"] == args.queries:
                    dram = tr["dram_bytes_read_per_launch"] + tr["dram_bytes_write_per_launch"]
                    traffic = {"dram_bytes_per_launch": dram, "algorithmic_bytes_per_launch": int(algo_bytes / n_launch),
                               "ratio": dram / (algo_bytes / n_launch), "source": tr["source"]}
                    break
            except Exception:
                pass
        cfg = base_config(args)
        line = {
            "metric": "GCUPS (score-only SW)", "value": gcups, "unit": "GCUPS", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_s / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": arith,
            "data": "synthetic", "config": cfg,
            "detail": {"kernel": kname, "wall_ms_per_step": wall_s / args.steps * 1e3, "checksum": checksum},
            "roofline": {"bound": "int_pipe", "achieved": per_gpu, "peak": pipe_gcups, "unit": "GCUPS",
                         "frac": per_gpu / pipe_gcups,
                         "peak_def": f"ALU-pipe bound of this kernel: 148 SM x {pk['sm_max_mhz']:.0f} MHz x R_int {r_int:.2f} "
                                     f"thread-instr/clk/SM (measured, {PIPE_PROFILE}) x 2 cells / {alu_per_pair} ALU-pipe instr "
                                     f"per cell pair ({alu_src}); the recurrence's adds co-issue on the FMA-side pipe",
                         "issue_slots_per_cell_pair": issue_per_pair,
                         "survey_frac": per_gpu / survey_gcups, "survey_peak": survey_gcups,
                         "survey_def": "SURVEY 8(d): same peak with 6 integer-pipe instr per 2 cells; > 1 because the kernel "
                                       "evaluates an algebraically equivalent 3.5-instruction form (DESIGN.md section 2), "
                                       "checked against the CPU oracle inside this run",
                         "traffic": traffic,
                         "hbm": {"algorithmic_bytes_per_step": int(algo_bytes),
                                 "achieved_gbs": algo_bytes / (dev_s / args.steps) / 1e9,
                                 "peak_gbs": pk["hbm_gbs"], "peak_source": pk["source"],
                                 "frac": algo_bytes / (dev_s / args.steps) / 1e9 / pk["hbm_gbs"]}},
            "cpu_baseline": cpu, "e2e": e2e, "single_handle": single,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        line.update(extra)
        emit(line)
    try:
        eng.close()
    except Exception:
        pass
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
