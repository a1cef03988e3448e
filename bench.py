#!/usr/bin/env python
"""bench.py -- GCUPS of the database-search hot path on N B200s, beside the reference on host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload config3|config2]
                  [--dump-outputs DIR]

Default workload = BASELINE.json configs[2], the largest single-GPU configuration: the 20 customary query
lengths 144 ... 5478 in the modes NW, HW and OV (score + end location) against the synthetic 570k-sequence /
207 M-residue Swiss-Prot-shaped database, BLOSUM62, gaps 11/1 -- the reference's own performance protocol, modes x
queries over one big database (reference test/perf:15-24), timed like the reference times it (the search call only,
src/opal_aligner.cpp:157-165) and scored with its formula, GCUPS = queryLength * sum(dbSeqLengths) / 1e9 / seconds
(src/opal_aligner.cpp:205-206).  A STEP is one sweep of that set: 60 searches, 25.9 T cell updates.  With N > 1 (one
process per GPU under torchrun) the database is dealt residue-balanced over the ranks (STRONG scaling; targets are
independent, so there is no data-path collective) and every rank runs the same 60 searches against its shard.

  value  device-timed: CUDA events on the library's streams, start of a batch of queries to its last kernel end,
         database resident in HBM, summed over the steps, max over ranks.
  e2e    the same sweep through the reference-facing C ABI call opalSearchDatabase, one call per (query, mode) with
         HOST buffers: database packing, H2D, kernels, D2H and the per-record result writes are all inside its
         timed region, every call.

`--workload config2` is BASELINE configs[1] (SW score+end, P18080 vs 12,071 sequences; weak scaling, one shard of
equal work per GPU) -- the headline of round 1, kept as a secondary measurement.
`--shard-of M` (development) runs rank 0's shard of an M-way deal on one GPU: the per-GPU time of an M-GPU run.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Searches in flight use streams of their own; with the default 8 hardware queues unrelated streams wait for each
# other's launches (libopal_b200.so sets this itself when it is loaded first; here torch initialises CUDA before it).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from opal_b200 import (MODES, OPAL_OVERFLOW_BUCKETS, OPAL_SEARCH_SCORE, OPAL_SEARCH_SCORE_END, OpalCLibrary,  # noqa: E402
                       SequenceDB, datasets, matrices, new_results, result_pointers, sharding)

GAP_OPEN, GAP_EXT = 11, 1
CPU_MAX_TARGET = 20000  # the reference's NW/HW/OV 32-bit pass is undefined behaviour (SURVEY.md 8c Q1): keep it out of the CPU sample


# ----------------------------------------------------------------------------- workloads
class Workload:
    pass


def make_workload(name, rank, world, shard_of=0):
    w = Workload()
    w.name, w.sm = name, matrices.blosum62()
    sm = w.sm
    p18080 = sm.encode(datasets.P18080)
    if name == "config2":
        # weak scaling: every GPU gets a shard of exactly the same work -- the same lengths and planted homologs, the
        # background residues redrawn per rank -- so that the per-GPU tail (the longest target) does not vary by rank
        w.db = datasets.config2_db(sm, p18080, residue_seed=None if rank == 0 else 20261017 + rank)
        w.full_sequences, w.full_residues = len(w.db) * world, None
        w.queries, w.modes, w.search_type = [p18080], ["SW"], OPAL_SEARCH_SCORE_END
        w.desc = ("BASELINE configs[1]: SW score+end, P18080 (Q=513) vs synthetic 12,071-seq Swiss-Prot-shaped DB, "
                  "BLOSUM62 11/1; one such shard per GPU (same lengths, residues redrawn per rank)")
        w.scaling = "weak"
    elif name == "config3":
        full = datasets.config3_db(sm, query=p18080)
        w.full_sequences, w.full_residues = len(full), full.total_residues
        parts = shard_of if shard_of > 1 else world
        w.db = sharding.shard_db(full, sharding.deal_shards(full.lengths, parts)[rank if shard_of <= 1 else 0]) if parts > 1 else full
        w.full_db = full
        w.queries = sorted(datasets.config3_queries(sm), key=len, reverse=True)  # longest first: the batch ends on short tails
        w.modes, w.search_type = ["NW", "HW", "OV"], OPAL_SEARCH_SCORE_END
        w.desc = ("BASELINE configs[2]: NW/HW/OV score+end, the 20 query lengths 144..5478 (sum 41,752) vs synthetic "
                  "570k-seq / 207M-residue Swiss-Prot-shaped DB with a heavy tail up to 35,213, BLOSUM62 11/1; one step = "
                  "60 searches (reference test/perf protocol); DB dealt residue-balanced over the GPUs")
        w.scaling = "strong"
    else:
        raise SystemExit(f"unknown workload {name}")
    w.sum_q = int(sum(len(q) for q in w.queries))
    return w


def config_of(w):
    """The `config` object: identical in both arms (same workload, same keys)."""
    return {"workload": w.desc, "modes": w.modes, "search": "score+end", "query_lengths": sorted(len(q) for q in w.queries),
            "matrix": "BLOSUM62", "gap_open": GAP_OPEN, "gap_ext": GAP_EXT, "db_sequences": w.full_sequences}


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.ok = [], set(), False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        for bit, name in names.items():
            if r & bit:
                self.reasons.add(name)

    def _loop(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.02)

    def start(self):
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        self.thread.join()
        self.sample()
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_library():
    ref = os.path.join(ROOT, "oracle", "_ref", "libopal_ref.so")
    if os.path.exists(ref):
        return OpalCLibrary(ref), "reference"
    port = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(port):
        import subprocess
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return OpalCLibrary(port), "port"


def cpu_sweep(lib, w, shards):
    """One sweep (every mode x every query) against all shards, one host thread per shard (the reference is
    re-entrant; ctypes releases the GIL).  Returns wall seconds."""
    sm = w.sm
    results = [new_results(len(s)) for s in shards]
    blank = [r.copy() for r in results]
    ptrs = [result_pointers(r) for r in results]
    rcs = [0] * len(shards)

    def work(k):
        for mode in w.modes:
            for q in w.queries:
                np.copyto(results[k].view(np.uint8), blank[k].view(np.uint8))
                rc, _ = lib.search_database(q, shards[k], GAP_OPEN, GAP_EXT, sm.flat(), sm.alphabet_length, results[k],
                                            w.search_type, MODES[mode], OPAL_OVERFLOW_BUCKETS, result_ptrs=ptrs[k])
                rcs[k] |= rc

    threads = [threading.Thread(target=work, args=(k,)) for k in range(len(shards))]
    t0 = time.perf_counter()
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    dt = time.perf_counter() - t0
    assert all(rc == 0 for rc in rcs), rcs
    return dt


def split_for_threads(db, nthreads, stride=1, max_len=None):
    """Contiguous residue-balanced shards of every `stride`-th sequence of the length-sorted DB."""
    order = np.argsort(db.lengths, kind="stable")
    if max_len is not None:
        order = order[db.lengths[order] <= max_len]
    order = order[::stride]
    lens = db.lengths[order].astype(np.int64)
    bounds = np.searchsorted(np.cumsum(lens), np.linspace(0, lens.sum(), nthreads + 1)[1:-1])
    parts = np.split(order, bounds)
    return [db.subset(p) for p in parts if len(p)], int(lens.sum())


def cpu_sample(w, db, seconds):
    """Shards of a stratified sample of `db` sized for about `seconds` of host work per sweep (assuming ~4 GCUPS per
    host thread, the order of what the AVX2 reference reaches in these modes)."""
    cores = os.cpu_count() or 1
    cells = float(w.sum_q) * len(w.modes) * db.total_residues
    stride = max(1, int(np.ceil(cells / (seconds * 4e9 * cores))))
    shards, residues = split_for_threads(db, cores, stride, CPU_MAX_TARGET if w.name == "config3" else None)
    note = (f"every {stride}-th sequence of the length-sorted DB" + (f" among those <= {CPU_MAX_TARGET} residues" if w.name == "config3" else "")
            + f" ({residues} residues), {len(w.modes) * len(w.queries)} searches per sweep, one std thread per contiguous residue-balanced shard")
    return shards, residues, note


def run_reference_arm(args, rank):
    if rank != 0:
        return
    w = make_workload(args.workload, 0, 1)
    lib, kind = cpu_library()
    shards, residues, note = cpu_sample(w, w.db, 4.0)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_sweep(lib, w, shards)
    secs = sum(cpu_sweep(lib, w, shards) for _ in range(args.steps))
    cells = float(w.sum_q) * len(w.modes) * residues * args.steps
    value = cells / 1e9 / secs
    line = {"impl": "reference", "metric": "GCUPS", "value": value, "unit": "GCUPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3,
            "higher_is_better": True, "scaling": w.scaling, "vs_baseline": None,
            "dtype": "int8/int16/int32 (AVX2)" if kind == "reference" else "int64",
            "data": "synthetic", "config": config_of(w),
            "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": len(shards), "kind": kind, "sample": note + ", per step"},
            "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- output dump
DUMP_TARGETS = 32768  # 60 searches x 3 arrays x 32,768 targets in float64 = 47 MB: a dump stays under 64 MB
DUMP_UNWRITTEN = np.iinfo(np.int32).min  # in a dump: an entry the last step did not write (no score or location)


def dump_outputs(path, arrays, n):
    """Writes the result arrays of the last timed step as <path>/<name>.npy in float64 (int32 values, exact), for
    comparing two builds output for output.  A database of more than DUMP_TARGETS targets is sampled: the same seeded
    choice of target indices every run, written beside them as target_index.npy.  Rows of a batch are the searches in
    the order they were issued."""
    cols = np.arange(n)
    if n > DUMP_TARGETS:
        cols = np.sort(np.random.default_rng(0).choice(n, DUMP_TARGETS, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "target_index.npy"), cols.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a[..., cols].astype(np.float64))


# ----------------------------------------------------------------------------- B200 arm
def run_b200_arm(args, rank, local_rank, world):
    import torch
    from opal_b200.handle import OpalB200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; opal-b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    os.environ["OPAL_B200_DEVICE"] = str(local_rank)  # device of the drop-in entry points (they take no device argument)
    # one process per GPU on one host: the library's host pool (packing, result scatter) gets this rank's share of the cores
    os.environ.setdefault("OPAL_B200_HOST_THREADS", str(max(1, (os.cpu_count() or 1) // max(world, 1))))
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    eng = OpalB200()
    w = make_workload(args.workload, rank, world, args.shard_of)
    sm, db = w.sm, w.db
    mat, A = sm.flat(), sm.alphabet_length
    handle = eng.create_db(db, local_rank)
    cells_rank = float(w.sum_q) * len(w.modes) * db.total_residues  # per step
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    single = len(w.queries) == 1
    nq, n = len(w.queries), len(db)
    # the searches of one step, in the order they are issued: query by query (longest first), its modes back to back;
    # "interleave" alternates long and short queries, so that the long single-warp tails of short queries (a 35k-residue
    # target costs the same steps whatever the query) run beside the bulk of long ones
    order = list(range(nq))
    if args.order == "interleave":
        order = [order[k // 2] if k % 2 == 0 else order[nq - 1 - k // 2] for k in range(nq)]
    searches = [(w.queries[k], mode) for k in order for mode in w.modes]
    out = None if single else tuple(np.zeros((len(searches), n), dtype=np.int32) for _ in range(3))
    last = {}  # what the latest step returned to its caller: score, end in query, end in target

    def step_resident():
        """One sweep against the resident database; returns (device ms, kernel launches)."""
        flush.zero_()
        torch.cuda.synchronize()
        if single:
            rc, sc, eq, et, ms = handle.search(w.queries[0], GAP_OPEN, GAP_EXT, mat, A, w.search_type, w.modes[0])
        else:  # one batch: every (query, mode) of the step, several in flight
            rc, sc, eq, et, ms = handle.search_batch([q for q, _ in searches], GAP_OPEN, GAP_EXT, mat, A, w.search_type,
                                                     [m for _, m in searches], in_flight=args.in_flight, out=out)
        if rc != 0:
            raise SystemExit(f"search failed rc={rc}: {eng.last_error()}")
        last.update(score=sc, end_query=eq, end_target=et)
        return ms, handle.last_stats()["kernel_launches"]

    # ---- device-timed value (database resident)
    for _ in range(args.warmup):
        step_resident()
    clocks = ClockSampler(local_rank)
    barrier()
    clocks.start()
    wall0 = time.perf_counter()
    dev_ms, launches, untimed = 0.0, 0, 0.0
    for step in range(args.steps):
        if args.dump_outputs and out is not None and step == args.steps - 1:
            # the batch keeps old values where it computes nothing: a sentinel makes the dump show only the last step
            t0 = time.perf_counter()
            for a in out:
                a.fill(DUMP_UNWRITTEN)
            untimed += time.perf_counter() - t0
        ms, ln = step_resident()
        dev_ms += ms
        launches += ln
    barrier()
    wall_resident = time.perf_counter() - wall0 - untimed
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, n)
    t_dev = reduce(dev_ms / 1e3, "MAX")
    t_wall = reduce(wall_resident, "MAX")
    total_cells = reduce(cells_rank, "SUM") * args.steps
    value = total_cells / 1e9 / t_dev
    check = None
    if not single:  # kept for the cross-check with the drop-in path below: the shortest query in the last mode
        k = max(i for i, (q, m) in enumerate(searches) if m == w.modes[-1] and len(q) == len(w.queries[-1]))
        check = out[0][k].copy()

    # ---- end to end through the drop-in C ABI (host buffers in, OpalSearchResult records out), one call per search
    blank = new_results(n)
    res = blank.copy()
    res_bytes, blank_bytes = res.view(np.uint8), blank.view(np.uint8)  # flat views: the reset below is one memcpy
    res_ptrs = result_pointers(res)  # the OpalSearchResult* array a C caller holds

    def step_e2e():
        for mode in w.modes:
            for q in w.queries:
                np.copyto(res_bytes, blank_bytes)  # the caller's opalInitSearchResult loop (reference src/opal_aligner.cpp:150-154)
                rc, _ = eng.search_database(q, db, GAP_OPEN, GAP_EXT, mat, A, res, w.search_type, MODES[mode], OPAL_OVERFLOW_BUCKETS,
                                            result_ptrs=res_ptrs)
                if rc != 0:
                    raise SystemExit(f"opalSearchDatabase failed rc={rc}: {eng.last_error()}")

    step_e2e()
    if check is not None:
        assert (res["score"] == check).all(), "drop-in call and resident handle disagree"
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    t_e2e = reduce(time.perf_counter() - t0, "MAX")
    e2e_value = total_cells / 1e9 / t_e2e
    # per call: one upload block [offsets | pair offsets | fold offsets | lengths | max code | residues] + one argument
    # block [counters | matrix | query]; three result arrays come back
    n_fold = max(min(n & ~1, 128), 1)
    index_bytes = (8 * (n + 1) + 8 * max((n + 1) // 2, 1) + 8 * n_fold + 4 * (max(n, 1) + 1) + 255) // 256 * 256
    calls = len(w.modes) * nq
    h2d = int(calls * (index_bytes + db.total_residues + 64 + 1024 + (4 * A * A + 255) // 256 * 256 + 16) + len(w.modes) * w.sum_q)
    d2h = int(calls * (3 * 4 * n + 4))

    # ---- one process, every GPU (N > 1): the same sweep as ONE opalSearchDatabase call per search over the WHOLE database,
    # dealt over all N devices inside the library (OPAL_B200_DEVICES); rank 0 alone, the other ranks wait on the host
    one_process = None
    if world > 1 and not single and not args.no_extras:
        import datetime
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            full = w.full_db
            os.environ["OPAL_B200_DEVICES"] = ",".join(str(d) for d in range(world))
            blank_full = new_results(len(full))
            res_full = blank_full.copy()
            rf_bytes, bf_bytes = res_full.view(np.uint8), blank_full.view(np.uint8)
            rf_ptrs = result_pointers(res_full)

            def sweep_all_devices():
                for mode in w.modes:
                    for q in w.queries:
                        np.copyto(rf_bytes, bf_bytes)
                        rc, _ = eng.search_database(q, full, GAP_OPEN, GAP_EXT, mat, A, res_full, w.search_type, MODES[mode], OPAL_OVERFLOW_BUCKETS,
                                                    result_ptrs=rf_ptrs)
                        if rc != 0:
                            raise SystemExit(f"opalSearchDatabase on {world} devices failed rc={rc}: {eng.last_error()}")

            sweep_all_devices()
            t0 = time.perf_counter()
            sweep_all_devices()
            dt = time.perf_counter() - t0
            del os.environ["OPAL_B200_DEVICES"]
            one_process = {"value": float(w.sum_q) * len(w.modes) * full.total_residues / 1e9 / dt, "unit": "GCUPS", "devices": world,
                           "ms_per_step": dt * 1e3,
                           "note": "wall clock, one process: each opalSearchDatabase call packs, uploads and searches the whole database on all "
                                   "devices (host threads of this process: its 1/N share of the cores, as for the e2e figure)"}
            store.set("one_process_done", "1")
        else:
            store.wait(["one_process_done"], datetime.timedelta(seconds=1800))

    # ---- extras (rank 0's shard, untimed region): every (mode, query) alone, score+end and score only; SW beside them
    extras = {}
    if rank == 0 and not single and not args.no_extras:
        per_query = {}
        for mode in w.modes + ["SW"]:
            for st, key in ((OPAL_SEARCH_SCORE_END, "score+end"), (OPAL_SEARCH_SCORE, "score")):
                row = {}
                for q in sorted(w.queries, key=len):
                    best = None
                    for _ in range(2):  # best of two: the first use of a kernel variant includes loading it
                        rc, _, _, _, ms = handle.search(q, GAP_OPEN, GAP_EXT, mat, A, st, mode)
                        if rc != 0:
                            raise SystemExit(f"search failed rc={rc}: {eng.last_error()}")
                        best = ms if best is None else min(best, ms)
                    row[str(len(q))] = round(len(q) * db.total_residues / 1e6 / best, 1)
                per_query[f"{mode} {key}"] = row
        extras["per_query_gcups_one_gpu"] = {
            "note": "single searches on rank 0's shard, device-timed first launch to last kernel end, GCUPS of one GPU by query length",
            "table": per_query}

    # ---- roofline of the dominant kernel class: packed-DPX issue rate (measured live) and HBM streaming
    global_modes = all(m != "SW" for m in w.modes)
    peak_gcups, instr_per_s, _ = eng.measure_dpx_peak(local_rank, mix=1 if global_modes else 0)
    per_gpu = value / world
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm_peak = float(json.load(f)["hbm_gbs"])
        hbm_src = "measured (MEASURED_PEAKS.json)"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    hbm_gbs = db.total_residues * calls * args.steps / (dev_ms / 1e3) / 1e9
    instr = 5 if global_modes else 6
    roofline = {
        "bound": "dpx (integer pipe)", "achieved": per_gpu, "peak": peak_gcups, "unit": "GCUPS", "frac": per_gpu / peak_gcups,
        "traffic": None,
        "traffic_note": "not measurable in-run; dram__bytes of the bulk launches are in the committed ncu --set full captures "
                        "(profiles/README.md): traffic = algorithmic bytes, DRAM < 1 % busy",
        "achieved_note": "whole step (all launches, tails and launch gaps included) per GPU; algorithmic work = "
                         f"{instr} packed s16x2 instructions per 2 cells ({'NW/HW/OV' if global_modes else 'SW'} recurrence, SURVEY.md 8d)",
        "peak_source": f"measured live: {instr_per_s / 1e12:.2f} T packed s16x2 thread-instr/s x 2 cells / {instr} instr",
        "hbm": {"bound": "hbm", "achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                "peak_source": hbm_src, "note": "algorithmic bytes = 1 B per DB residue per query (1/Q B per cell)"},
    }

    line = None
    if rank == 0:
        stats = handle.last_stats()
        line = {"metric": "GCUPS", "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": w.scaling, "vs_baseline": None,
                "dtype": "s16x2 (DPX), s32 where 16 bits cannot hold the scores", "data": "synthetic",
                "config": config_of(w),
                "details": {"db_sequences_per_gpu": n, "db_residues_per_gpu": db.total_residues,
                            "cells_per_step": total_cells / args.steps, "queries_in_flight": 1 if single else args.in_flight,
                            "query_order": args.order,
                            "l2": "256 MiB flush buffer written between timed steps",
                            "wall_ms_per_step_resident": t_wall / args.steps * 1e3,
                            "last_geometry": {k: stats[k] for k in ("G", "R", "passes", "warps_per_partition", "groups", "folded")}},
                "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": t_e2e / args.steps * 1e3,
                        "path": f"opalSearchDatabase x {calls} per step (each: pack + H2D + kernels + D2H + records)"},
                "gpu_launches": launches, "clocks": clk, "roofline": roofline}
        if args.shard_of > 1:
            line["details"]["emulation"] = f"rank 0's shard of a {args.shard_of}-way deal on one GPU (development run, not a scaling result)"
        line.update(extras)
        if one_process:
            line["one_process_multi_gpu"] = one_process

    # ---- CPU baseline beside it (rank 0, N = 1 only)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        lib, kind = cpu_library()
        shards, residues, note = cpu_sample(w, w.full_db if hasattr(w, "full_db") else db, 4.0)
        cpu_sweep(lib, w, shards)
        reps, secs = 0, 0.0
        while secs < 12.0 and reps < 200:
            secs += cpu_sweep(lib, w, shards)
            reps += 1
        line["cpu_baseline"] = {"value": float(w.sum_q) * len(w.modes) * residues * reps / 1e9 / secs, "unit": "GCUPS",
                                "cores": len(shards), "kind": kind, "sample": note + f", x {reps} sweeps"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    handle.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config3", choices=["config2", "config3"])
    ap.add_argument("--in-flight", type=int, default=12, help="queries of a batch on the device at a time")
    ap.add_argument("--order", default="desc", choices=["desc", "interleave"], help="order of the queries within a step")
    ap.add_argument("--shard-of", type=int, default=0, help="development: run one shard of an M-way deal on one GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy "
                    "(rank 0's shard; float64, a fixed sample of the targets of a large database)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the B200 arm (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args, rank)
    else:
        run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
