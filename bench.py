#!/usr/bin/env python
"""bench.py -- GCUPS of the ssw_align hot path (BASELINE.json metric) on the named shapes.

  python bench.py --gpus N --steps K --warmup W          our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W  the reference's own SSE2 path on the host cores
  python bench.py ... --dump-outputs DIR                  also write the records of every shape's last timed step (dump_outputs)

Headline workload (BASELINE.json configs[2], SURVEY 8(d) "config 3", the shape north_star's scaling target is quoted on):
100,000 synthetic 150 bp DNA reads x one 5 Mbp reference, DNA matrix 2/-2 (N = 0), gap open 3 / extend 1, score_size 2
(byte pass, word re-run on overflow), flag 0, maskLen 75.  STRONG scaling: the one pair list is cut into cell-balanced
contiguous shards (ssw_dist.shard_range; the reference's loop being sharded is main.c:462-532), every rank aligns its
shard on its own GPU, and the records are gathered to rank 0 over NCCL -- inside the timed region.
GCUPS = sum(readLen * refLen) / time / 1e9, cells counted once per pair.

The same line carries the other named shapes as sub-results ("config2", "config4", "config5"), each with its own
device-resident rate, end-to-end rate, per-phase times, ALU roofline and (N = 1) CPU rate for the same shape, and an
untimed parity self-check of gathered records against the compiled reference (oracle/_ref/libssw_ref.so; checker only).

`value`: sequences already resident in HBM when the timed region starts.  `e2e`: host buffers through the C ABI
(ssw_engine_set_sequences: H2D of every sequence; ssw_engine_align: kernels + D2H of the records) + the gather to rank 0.
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written there, not even __pycache__
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ALG_BYTES_NOTE = "refLen + readLen + n*n + 40 bytes per pair (SURVEY 8(d))"
METRIC = "GCUPS (DP cell updates/s), ssw_align forward path"
CONFIG_NOTES = {
    "l2": "b200 arm: a 256 MB buffer is written between timed steps (L2 flush) and every step streams its own scratch; reference arm: CPU, n/a",
    "timing": "b200 arm: per step max(CUDA-event time on the engine stream, wall clock between synchronised barriers), max over ranks; "
              "reference arm: wall clock of the pthread harness over a bounded sample of the same read set (a rate)",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=100_000, help="reads of the headline batch (config 3: 100,000)")
    ap.add_argument("--only", default="3,2,4,5", help="shapes to run, e.g. 3,2 (3 is the headline and always runs)")
    ap.add_argument("--e2e-reps", type=int, default=2, help="timed end-to-end repetitions per shape")
    ap.add_argument("--sub-steps", type=int, default=3, help="timed steps of the sub-result shapes (configs 2, 4, 5)")
    ap.add_argument("--c4-queries", type=int, default=512, help="queries of the config-4 slice (of 10,000) x all 50,000 targets")
    ap.add_argument("--c4-targets", type=int, default=50_000)
    ap.add_argument("--parity", type=int, default=256, help="gathered config-3 records re-computed by the CPU reference (untimed)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the CPU sample of the headline shape (0: 8 per usable core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--opt", action="append", default=[], help="experiment: engine option name=value (repeatable)")
    ap.add_argument("--clock-sampler", choices=["smi", "nvml"], default="smi",
                    help="how clocks / throttle reasons are sampled during the timed region")
    ap.add_argument("--lib", default="libssw.so", help="experiment: alternative build of the library")
    ap.add_argument("--dry-run-emu", action="store_true",
                    help="tests only: run the orchestration on the CPU emulator build of the kernels (tests/cuda_emu) with tiny shapes and "
                         "the gloo backend; the printed line is marked dry_run and its numbers mean nothing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the records (and CIGAR words) the last timed step of every shape returned as "
                         "DIR/<shape>_<field>.npy, float64 (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.sub_steps < 1:
        ap.error("--steps and --sub-steps must be at least 1")
    return args


def workload_name(n_reads):
    return ("config3: %d x 150 bp reads vs one 5000000 bp reference, byte-score path with word re-run on overflow, flag 0, maskLen 75; "
            "one pair list sharded over the GPUs (cell-balanced contiguous blocks), records gathered to rank 0" % n_reads)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class NvmlSampler:
    """The same quantities read in-process through NVML (nvidia_ml_py) every 100 ms: no nvidia-smi process polling the
    driver while the timed region runs."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.h = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.idx
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.h = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml unavailable"}
        bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        seen = 0
        for r in self.rows:
            seen |= int(r[2])
        return {"sm_mhz": float(np.median([r[0] for r in self.rows])), "sm_max_mhz": float(max(r[1] for r in self.rows)),
                "reasons": sorted(k for k, b in bits.items() if seen & b), "samples": len(self.rows), "source": "nvml, 100 ms period"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores (oracle/_ref; checker / baseline only)
# ------------------------------------------------------------------------------------------------

def cpu_rate(W, pair_q, pair_r, threads):
    """GCUPS of the CPU implementation (compiled reference if present, else the scalar port) on the given pairs of
    workload W with `threads` pthreads (oracle/ssw_harness.c).  Returns (gcups, kind, seconds, records, pool)."""
    import common as C
    rec, pool, secs, cells, kind = C.cpu_batch(W["queries"], W["refs"], pair_q, pair_r, W["mat"], W["n"], W["gapO"], W["gapE"], W["flag"],
                                               W["filters"], W["filterd"], W["mask_len"], W["score_size"], threads=threads)
    return cells / secs / 1e9, kind, secs, rec, pool


def cpu_baseline_obj(W, pair_q, pair_r, what):
    import common as C
    cores, info = C.effective_cores()
    v, kind, secs, _, _ = cpu_rate(W, pair_q, pair_r, cores)
    return {"value": v, "unit": "GCUPS", "cores": cores, "kind": kind, "gcups_per_thread": v / cores,
            "sample": "%s, %d pthreads (oracle/ssw_harness.c), %.1f s" % (what, cores, secs),
            "cores_detail": info}


def run_reference(args):
    """--impl reference: the reference's CPU implementation on all usable host cores; rank 0 only.  Each step aligns a
    bounded sample (the first reads of the same 100,000-read set) and reports the rate."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import common as C
    cores, info = C.effective_cores()
    sample = args.cpu_sample or 8 * cores
    if not C.have_ref():
        sample = max(2, cores // 4)          # the scalar port is ~20x slower than SSE2
    W = C.config_workload(3, n_reads=sample)        # the generator is sequential: these ARE the first reads of the full set
    pq, pr = np.arange(sample), np.zeros(sample)
    vals = []
    kind = "reference"
    for s in range(args.warmup + args.steps):
        v, kind, dt, _, _ = cpu_rate(W, pq, pr, cores)
        if s >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "GCUPS",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8 (SSE2 16-lane saturating), i16 re-run on overflow", "data": "synthetic",
            "config": dict(workload=workload_name(args.reads), **CONFIG_NOTES),
            "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": cores, "kind": kind, "gcups_per_thread": value / cores,
                             "sample": "each step: the first %d reads of the %d-read set x the 5 Mbp reference on %d pthreads (a rate; the full batch is ~%.0f CPU-hours)"
                                       % (sample, args.reads, cores, args.reads * 7.5e8 / (value * 1e9 / cores) / 3600.0),
                             "cores_detail": info},
            "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------

class Ctx:
    pass


def shard_of(W, cfg, D, rank, world):
    """This rank's block of the work: reads (configs 2, 3, 5; cell-balanced) or queries of the grid (config 4)."""
    qs = W["queries"]
    if cfg == 4:
        return D.split_even(len(qs), rank, world)
    cells = [len(q) * len(W["refs"][0]) for q in qs]
    return D.shard_range(cells, rank, world)


def run_shape(X, cfg, W, steps, warmup, e2e_reps, sampler=None, dump=None):
    """Time one shape.  Returns (stats dict on every rank, gathered records + pool on rank 0).  dump: called on rank 0 with
    what the last timed step returned, before the end-to-end repetitions re-use its buffers."""
    import torch
    import torch.distributed as dist
    D, L, eng = X.D, X.L, X.eng
    lo, hi = shard_of(W, cfg, D, X.rank, X.world)
    mine = W["queries"][lo:hi]
    refs = W["refs"]
    n_q_all, n_r = len(W["queries"]), len(refs)
    cells_total = float(sum(len(q) for q in W["queries"])) * float(sum(len(r) for r in refs))
    kw = dict(flag=W["flag"], filters=W["filters"], filterd=W["filterd"], mask_len=W["mask_len"], score_size=W["score_size"])
    dev = X.dev

    def barrier():
        if X.world > 1:
            dist.barrier()
        if not X.emu:
            torch.cuda.synchronize()

    keep = {"res": None}

    def step_resident():
        res, pool = eng.align(W["mat"], W["n"], W["gapO"], W["gapE"], out=keep["res"], **kw)     # the caller's record buffer is re-used
        keep["res"] = res
        return D.gather_batch(res, pool, X.rank, X.world, device=dev)

    def step_e2e():
        eng.set_sequences(mine, refs)                      # H2D of this rank's sequences (pageable host buffers)
        return step_resident()

    eng.set_sequences(mine, refs)
    for _ in range(warmup):
        step_resident()
    if sampler is not None and X.rank == 0:
        sampler.start()
    acc = {k: 0.0 for k in ("total_ms", "fill_forward_ms", "resolve_ms", "fill_reverse_ms", "traceback_ms")}
    launches = fill_launches = overflows = 0
    wall = 0.0
    got = None
    for _ in range(steps):
        X.flush.zero_()                       # flush L2 between timed iterations (untimed)
        barrier()
        t0 = time.perf_counter()
        got = step_resident()
        barrier()
        wall += time.perf_counter() - t0
        tm = eng.timing()
        for k in acc:
            acc[k] += tm[k]
        launches += tm["fill_forward_launches"] + tm["other_launches"]
        fill_launches += tm["fill_forward_launches"]
        overflows = tm["byte_overflows"]
    clocks = sampler.stop() if (sampler is not None and X.rank == 0) else None
    if dump is not None and X.rank == 0:
        dump(got)
    tt = torch.tensor([acc["total_ms"], wall * 1e3, acc["fill_forward_ms"], acc["resolve_ms"], acc["fill_reverse_ms"], acc["traceback_ms"]],
                      dtype=torch.float64, device=dev)
    cnt = torch.tensor([launches, fill_launches, overflows], dtype=torch.int64, device=dev)
    if X.world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    dev_ms, wall_ms, fill_ms, res_ms, rev_ms, tb_ms = [float(x) / steps for x in tt.tolist()]
    step_ms = max(dev_ms, wall_ms)               # the slower of the two clocks: never flatter than the driver's own
    launches, fill_launches, overflows = [int(x) for x in cnt.tolist()]

    # ---- end to end: host buffers -> C ABI -> records on rank 0 ----
    e2e_ms = None
    if e2e_reps > 0:
        step_e2e()
        e2e_wall = 0.0
        for _ in range(e2e_reps):
            X.flush.zero_()
            barrier()
            t0 = time.perf_counter()
            got = step_e2e()
            barrier()
            e2e_wall += time.perf_counter() - t0
        t = torch.tensor([e2e_wall / e2e_reps], dtype=torch.float64, device=dev)
        if X.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item()) * 1e3
    h2d = int(sum(len(q) for q in mine) + sum(len(r) for r in refs) + len(W["mat"]))
    n_pairs_rank = (hi - lo) * n_r
    step_ms = max(step_ms, 1e-6)
    stats = {"cells": cells_total, "step_ms": step_ms, "device_ms": dev_ms, "wall_ms": wall_ms,
             "value": cells_total / (step_ms * 1e-3) / 1e9,
             "e2e_ms": e2e_ms, "e2e_value": (cells_total / (e2e_ms * 1e-3) / 1e9) if e2e_ms else None,
             "fill_ms": fill_ms, "resolve_ms": res_ms, "reverse_ms": rev_ms, "traceback_ms": tb_ms,
             "launches_total": launches, "fill_launches_per_step_all_ranks": fill_launches / steps, "byte_overflows": overflows,
             "h2d_rank0": h2d, "d2h_rank0": int(36 * n_pairs_rank + (4 * len(got[1]) if (got and got[1] is not None and X.world == 1) else 0)),
             "pairs": n_q_all * n_r, "shard": [lo, hi], "clocks": clocks, "steps": steps, "warmup": warmup}
    return stats, got


DUMP_FIELDS = ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag", "status", "cigar_len")
DUMP_PAIRS = 1 << 18                     # records per shape at most: 10 fields x 8 bytes x 262,144 = 21 MB
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, shape, got):
    """rank 0: the records of the last timed step, one float64 array per field (DIR/<shape>_<field>.npy, pair order), and the
    CIGAR words of those pairs concatenated in pair order (DIR/<shape>_cigar.npy, written only when there are any: shapes run
    with flag 0 return no CIGAR; cigar_len splits them).  A shape with more
    than DUMP_PAIRS pairs is written as a fixed, seeded sample of them, whose pair indices go to DIR/<shape>_pair_index.npy.
    The inputs are seeded too, so two builds run with the same arguments can be compared array by array.  Returns the bytes
    written."""
    recs, pool = got
    pool = np.zeros(0, np.uint32) if pool is None else np.asarray(pool)
    idx = np.arange(len(recs))
    if len(recs) > DUMP_PAIRS:
        idx = np.sort(np.random.default_rng(0).choice(len(recs), DUMP_PAIRS, replace=False))
    arrays = {f: recs[f][idx].astype(np.float64) for f in DUMP_FIELDS}
    if len(idx) != len(recs):
        arrays["pair_index"] = idx.astype(np.float64)
    offs, lens = recs["cigar_off"][idx].astype(np.int64), recs["cigar_len"][idx].astype(np.int64)
    lens = np.where(offs < 0, 0, lens)
    starts = np.concatenate([[0], np.cumsum(lens)])
    if starts[-1] > 0:
        arrays["cigar"] = pool[np.repeat(offs - starts[:-1], lens) + np.arange(starts[-1])].astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, "%s_%s.npy" % (shape, name)), a)
    return sum(a.nbytes for a in arrays.values())


def parity_check(W, got, n_check, n_r):
    """rank 0, untimed: re-compute `n_check` gathered records, spread evenly over the whole pair list (so over every
    rank's shard), with the CPU reference and compare every field and every CIGAR word."""
    import common as C
    recs, pool = got
    n_pairs = len(recs)
    idx = np.unique(np.linspace(0, n_pairs - 1, min(n_check, n_pairs)).astype(np.int64))
    exp, exp_pool, secs, _, kind = C.cpu_batch(W["queries"], W["refs"], idx // n_r, idx % n_r, W["mat"], W["n"], W["gapO"], W["gapE"], W["flag"],
                                               W["filters"], W["filterd"], W["mask_len"], W["score_size"])
    bad = C.compare_records(recs, pool, exp, exp_pool, idx=idx)
    return {"parity_checked": int(len(idx)), "mismatches": int(len(bad)), "checker": kind, "seconds": round(secs, 1),
            "first_bad_pairs": [int(idx[i]) for i in bad[:4]]}


def alu_roofline(cells, fill_s):
    """Cell updates/s of the fill kernels against the measured DPX issue peak (profiles/dpx_peak.json, written by
    tools/microbench on the B200): 5.5 packed-s16x2 ops per 2 cells."""
    p = os.path.join(ROOT, "profiles", "dpx_peak.json")
    peak = None
    if os.path.exists(p):
        with open(p) as f:
            peak = json.load(f).get("gcups_peak_5p5_ops_per_cellpair")
    ach = cells / fill_s / 1e9 if fill_s > 0 else None
    return {"achieved_gcups": ach, "peak_gcups": peak, "frac": (ach / peak) if (peak and ach) else None,
            "unit": "GCUPS", "basis": "measured VIADDMNMX.S16x2 issue rate x 148 SMs / 2.75 ops per cell"}


def sub_result(st, world, name, what, extra=None):
    o = {"workload": what, "value": st["value"], "unit": "GCUPS", "ms_per_step": st["step_ms"], "steps": st["steps"], "warmup": st["warmup"],
         "e2e": {"value": st["e2e_value"], "unit": "GCUPS", "ms_per_step": st["e2e_ms"], "h2d_bytes_per_step_rank0": st["h2d_rank0"],
                 "d2h_bytes_per_step_rank0": st["d2h_rank0"]},
         "phases_ms": {"fill_forward": st["fill_ms"], "resolve": st["resolve_ms"], "fill_reverse": st["reverse_ms"], "traceback": st["traceback_ms"],
                       "note": "max over ranks, per step; phases of slices running on helper streams overlap, so they may add up to more than the step"},
         "alu_roofline": alu_roofline(st["cells"] / world, st["fill_ms"] * 1e-3), "pairs": st["pairs"], "byte_overflows": st["byte_overflows"]}
    if st["fill_ms"] > st["step_ms"]:
        # slices on helper streams: their fill times are taken while they share the device and add up to more than the step
        o["alu_roofline"] = alu_roofline(st["cells"] / world, st["step_ms"] * 1e-3)
        o["alu_roofline"]["basis"] += ("; denominator = the whole step (forward fills of concurrent slices overlap with reverse fills and tracebacks, "
                                       "their summed times exceed the step): a lower bound of the fill kernels' own efficiency "
                                       "(kernel alone: profiles/ncu_strips_cfg5_r2.txt)")
    if extra:
        o.update(extra)
    return o


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    import common as C
    from __graft_entry__ import load_package
    L = load_package()
    import importlib.util
    spec = importlib.util.spec_from_file_location("ssw_b200_dist", os.path.join(ROOT, "complete-striped-smith-waterman-library_b200", "ssw_dist.py"))
    D = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(D)

    X = Ctx()
    X.world = int(os.environ.get("WORLD_SIZE", "1"))
    X.rank = int(os.environ.get("RANK", "0"))
    X.local = int(os.environ.get("LOCAL_RANK", "0"))
    X.emu = args.dry_run_emu
    if X.emu:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cuda_emu")], check=True, stdout=sys.stderr)
        if X.world > 1:
            dist.init_process_group("gloo")
        X.dev = "cpu"
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(X.local)
        if X.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", X.local))
        X.dev = "cuda:%d" % X.local
    X.D, X.L = D, L
    X.eng = (L.BatchAligner(lib_dir=os.path.join(ROOT, "tests", "cuda_emu"), lib_name="libssw_emu.so") if X.emu
             else L.BatchAligner(device=X.local, lib_name=args.lib))
    if X.emu:
        X.eng.set_option("tb_spec", 0)          # the emulator runs warps one after the other: no point in speculative rounds
    for kv in args.opt:
        name, val = kv.split("=")
        X.eng.set_option(name, int(val))
    X.flush = torch.empty((1 << 10) if X.emu else (256 << 20), dtype=torch.uint8, device=X.dev)       # > 126 MB L2
    only = set(int(x) for x in args.only.split(",") if x.strip())
    rank0 = X.rank == 0
    do_cpu = rank0 and X.world == 1 and not args.no_cpu_baseline
    cores = C.effective_cores()[0]

    # ---- headline: config 3, strong-scaled ----
    tiny = dict(ref_len=2000, read_len=60) if X.emu else {}
    W3 = C.config_workload(3, n_reads=args.reads, **tiny)
    sampler = {"smi": ClockSampler, "nvml": NvmlSampler}[args.clock_sampler](X.local)
    dumped = []

    def dumper(shape):
        if args.dump_outputs:
            return lambda got: dumped.append(dump_outputs(args.dump_outputs, shape, got))
        return None

    st3, got3 = run_shape(X, 3, W3, args.steps, args.warmup, args.e2e_reps, sampler, dumper("config3"))
    line = None
    if rank0:
        hbm_peak, peak_src = peaks()
        n = W3["n"]
        ref_len = len(W3["refs"][0])
        alg_bytes_step = float(sum(ref_len + len(q) + n * n + 40 for q in W3["queries"])) / X.world      # per rank and step
        fl = max(st3["fill_launches_per_step_all_ranks"] / X.world, 1.0)                                  # launches per rank and step
        fill_s = max(st3["fill_ms"] * 1e-3, 1e-9)
        achieved = alg_bytes_step / fill_s / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic_fill.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            per_read = tj.get("dram_bytes_per_read")
            if per_read:
                traffic = float(per_read) * len(W3["queries"]) / X.world             # this rank's reads = one byte-pass launch
                traffic_src = ("static: %s B of DRAM traffic per read from the ncu capture of the 100,000-read launch (profiles/traffic_fill.json, %s) "
                               "x the reads of one launch; not measured in this run" % (per_read, tj.get("captured", "round 2")))
        line = {"metric": METRIC, "value": st3["value"], "unit": "GCUPS", "n_gpus": X.world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": st3["step_ms"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "s16x2 (byte- and word-score semantics in 16-bit DPX lanes)", "data": "synthetic",
                "config": dict(workload=workload_name(args.reads), **CONFIG_NOTES),
                "clocks": st3["clocks"],
                "e2e": {"value": st3["e2e_value"], "unit": "GCUPS", "ms_per_step": st3["e2e_ms"],
                        "h2d_bytes_per_step": st3["h2d_rank0"], "d2h_bytes_per_step": st3["d2h_rank0"],
                        "note": "per rank: ssw_engine_set_sequences (H2D of its reads + the reference, pageable host buffers) + ssw_engine_align "
                                "(kernels, D2H of the records) through the C ABI, then the NCCL gather of all records to rank 0; byte counts are rank 0's"},
                "gpu_launches": st3["launches_total"],
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                             "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes": ALG_BYTES_NOTE,
                             "kernel": "ssw_fill_kernel<8,20,+1> (forward fill: byte pass + word re-fill of the byte overflows)",
                             "kernel_ms_per_step": fill_s * 1e3, "kernel_launches_per_step_per_rank": fl,
                             "launch_accounting": "one step of a rank = one byte-pass launch over all its reads + one small word re-fill launch of the ~3 % byte overflows; "
                                                  "achieved / traffic / algorithmic bytes are for the rank's reads, the time is the sum of both launches",
                             "algorithmic_bytes_per_launch": alg_bytes_step,
                             "note": "integer-issue bound recurrence (150 cells per reference byte): the HBM fraction is reported as required, "
                                     "the meaningful efficiency is alu_roofline"},
                "alu_roofline": alu_roofline(st3["cells"] / X.world, fill_s),
                "phases_ms": {"fill_forward": st3["fill_ms"], "resolve": st3["resolve_ms"], "device_total": st3["device_ms"], "wall": st3["wall_ms"]},
                "byte_overflows": st3["byte_overflows"], "shards": "cell-balanced contiguous blocks of the read list (ssw_dist.shard_range)"}
        line["parity"] = {"config3": parity_check(W3, got3, args.parity, 1)}
        if do_cpu:
            sample = args.cpu_sample or 8 * cores
            if not C.have_ref():
                sample = max(2, cores // 4)
            sample = min(sample, len(W3["queries"]))
            line["cpu_baseline"] = cpu_baseline_obj(W3, np.arange(sample), np.zeros(sample), "the first %d reads of the set x the 5 Mbp reference" % sample)
    del got3

    # ---- sub-results: the other named shapes, same natural split ----
    subs = {}
    if 2 in only:
        W = C.config_workload(2, **(dict(n_reads=4, **tiny) if X.emu else {}))
        st, got = run_shape(X, 2, W, max(args.sub_steps, 3), 3, args.e2e_reps, dump=dumper("config2"))
        if rank0:
            o = sub_result(st, X.world, "config2", "1,000 x 150 bp reads vs 5 Mbp, byte-score path, flag 0 (strong: reads split over the GPUs)")
            ref_len = len(W["refs"][0])
            alg = float(sum(ref_len + len(q) + 25 + 40 for q in W["queries"])) / X.world
            hbm_peak, _ = peaks()
            fs = max(st["fill_ms"] * 1e-3, 1e-9)
            o["roofline"] = {"bound": "hbm", "achieved": alg / fs / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg / fs / 1e9 / hbm_peak, "kernel_ms_per_step": st["fill_ms"]}
            o["parity"] = parity_check(W, got, 64, 1)
            if do_cpu:
                sample = min(len(W["queries"]), 4 * cores)
                o["cpu_baseline"] = cpu_baseline_obj(W, np.arange(sample), np.zeros(sample), "%d of the 1,000 reads x 5 Mbp" % sample)
            subs["config2"] = o
    if 4 in only:
        W = C.config_workload(4, n_queries=args.c4_queries, n_targets=args.c4_targets)
        st, got = run_shape(X, 4, W, args.sub_steps, 2, args.e2e_reps, dump=dumper("config4"))
        if rank0:
            o = sub_result(st, X.world, "config4", "protein BLOSUM50, word-score path, flag 0: a %d-query slice of the 10,000 x 300 aa queries x all %d x 400 aa targets "
                           "(queries split over the GPUs, targets replicated; the full grid would return 18 GB of records)" % (args.c4_queries, args.c4_targets))
            o["parity"] = parity_check(W, got, 4096, len(W["refs"]))
            if do_cpu:
                rng = np.random.default_rng(7)
                k = 4000 * cores
                o["cpu_baseline"] = cpu_baseline_obj(W, rng.integers(0, len(W["queries"]), k), rng.integers(0, len(W["refs"]), k), "%d random pairs of the grid" % k)
            subs["config4"] = o
        del got
    if 5 in only:
        W = C.config_workload(5, **(dict(n_reads=3, ref_len=1500, read_len=330) if X.emu else {}))
        st, got = run_shape(X, 5, W, args.sub_steps, 2, args.e2e_reps, dump=dumper("config5"))
        if rank0:
            o = sub_result(st, X.world, "config5", "1,000 x 10 kbp reads vs 100 kbp, byte pass overflows -> word path, flag 2 (begin search + banded traceback, "
                           "CIGARs gathered in two phases: lengths, then payload)")
            o["cigar_words"] = int(len(got[1]))
            o["parity"] = parity_check(W, got, 24, 1)
            if do_cpu:
                sample = min(len(W["queries"]), max(cores, 8))
                o["cpu_baseline"] = cpu_baseline_obj(W, np.arange(sample), np.zeros(sample), "%d of the 1,000 reads x 100 kbp incl. CIGAR" % sample)
            subs["config5"] = o
    if rank0:
        line.update(subs)
        if X.emu:
            line["dry_run"] = "CPU emulator build, tiny shapes: numbers are meaningless"
        bad = line["parity"]["config3"]["mismatches"] + sum(s["parity"]["mismatches"] for s in subs.values())
        line["parity_checked"] = line["parity"]["config3"]["parity_checked"] + sum(s["parity"]["parity_checked"] for s in subs.values())
        line["mismatches"] = bad
        if args.dump_outputs:
            assert sum(dumped) <= DUMP_LIMIT, dumped
            line["dumped_bytes"] = sum(dumped)
        print(json.dumps(line))
    X.eng.close()
    if X.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
