#!/usr/bin/env python
"""bench.py -- headline benchmark of the pairwise-alignment hot path on B200.

Metric (BASELINE.json): GCUPS = sum over pairs of m*n / seconds / 1e9 (one cell update = T1, T2
and T3 of one (i, j); cells recomputed for traceback are not counted).

Headline workload at any N: BASELINE config 2 per GPU -- 1M synthetic 150 bp x 150 bp read pairs,
local (Smith-Waterman) score + end cell + traceback ops; even pairs mutated copies, odd pairs random
(seed 20250002 + rank).  Shards are independent: no data-path collective ("weak" scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned (see write_outputs), so that two builds can be compared
output for output on the same seeded inputs.

One JSON line on stdout (rank 0):
  value      device-resident inputs, CUDA-event timed, max over ranks
  e2e        the same pass through the host-buffer C-ABI call a production caller makes
             (psa_align_batch_packed: 2-bit fixed-stride reads in pinned host memory, H2D and D2H inside the
             timed region); `e2e_byte_api` = the same through psa_align_batch (raw bytes + offsets + lengths)
  roofline   the integer-issue roofline SURVEY 8(d) defines for this path, for the dominant kernel on its own
             launch durations (peak measured live by psa_peak_int_ops), plus the whole-step and HBM views
  cpu_baseline  the reference's own CPU implementation (oracle/_ref) on a bounded sample (N = 1 only)
  extra.configs sub-records for BASELINE configs 1, 3, 4, 5 (SURVEY 8d): GCUPS, roofline fraction and the CPU
             reference beside them at N = 1; at N > 1 config 4 runs as ONE pair split in column strips over
             the N GPUs and config 5 as 100 000 pairs sharded over them (strong scaling)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "GCUPS (cell updates/sec)"
READ_LEN = 150
OPS_LOCAL, OPS_GLOBAL = 7, 6      # SURVEY 8(d): 6 lane-ops per global cell, +1 running max for local
G, H = 1, 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=1_000_000, help="pairs per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 1/3/4/5 sub-records")
    ap.add_argument("--e2e-variants", action="store_true",
                    help="also time the end-to-end step with the chunk fills serialised or not x fixed-stride or compact ops")
    ap.add_argument("--extra-timeout", type=int, default=420, help="seconds the sub-records may take before the headline is printed without them")
    ap.add_argument("--c4-len", type=int, default=1_000_000)
    ap.add_argument("--c5-pairs", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; it cannot be combined with --impl reference")
    return args


def config_dict(args, world):
    return {"workload": "config2: batch of 1M synthetic 150bp x 150bp DNA read pairs, local SW score + traceback",
            "pairs_per_gpu": args.pairs, "read_len": READ_LEN, "mode": "local", "g": G, "h": H,
            "outputs": "score, end cell, start cell, 2-bit traceback ops",
            "parallelism": f"pair-shards x{world} (no collective)",
            "l2_policy": "inputs larger than L2 (300 MB of bases per step vs 126 MB L2)"}


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
def cpu_baseline(n_sample, seed, with_shipped=False, length=READ_LEN):
    """The reference's CPU implementation of the path, pair-parallel over all host cores
    (the shape of test_n_cores_thread, testing.cpp:269-276), best-case thread budget p=1 per pair
    plus the as-shipped p=32 call on a smaller sample.  kind 'reference' = oracle/_ref built from
    the reference's own sources; 'port' = the oracle restatement when _ref is absent."""
    from oracle import pyoracle as po
    from cse305_parallel_sequence_alignment_b200 import synth
    cores = os.cpu_count() or 1
    A, B = synth.read_pair_batch(n_sample, length, seed)
    off, ln = synth.fixed_length_layout(n_sample, length)
    a, b = np.ascontiguousarray(A.reshape(-1)), np.ascontiguousarray(B.reshape(-1))
    cells = float(n_sample) * length * length
    if po.have_ref():
        sec = po.ref_time_batch(a, off, ln, b, off, ln, 1, G, H, cores)
        out = {"value": cells / sec / 1e9, "unit": "GCUPS", "cores": cores, "kind": "reference",
               "sample": f"{n_sample} pairs of {length}x{length} through main_alignment_function(p=1), one pair per host "
                         f"thread x{cores}, global mode (the reference has no local mode; same cell count), "
                         f"built -O2, stdout to /dev/null",
               "seconds": sec}
        if with_shipped:   # the call exactly as the harness issues it: p=32 (testing.cpp:134)
            n32 = min(n_sample, cores)
            sec32 = po.ref_time_batch(a, off[:n32], ln[:n32], b, off[:n32], ln[:n32], 32, G, H, cores)
            out["as_shipped_p32_gcups"] = n32 * length * length / sec32 / 1e9
            out["as_shipped_sample_pairs"] = n32
        return out
    # port: thread the linear-space oracle over chunks (ctypes releases the GIL)
    chunks = np.array_split(np.arange(n_sample), cores)
    t0 = time.perf_counter()
    th = [threading.Thread(target=po.score_batch, args=(a, off[c], ln[c], b, off[c], ln[c], G, H, po.LOCAL)) for c in chunks if len(c)]
    [t.start() for t in th]
    [t.join() for t in th]
    sec = time.perf_counter() - t0
    return {"value": cells / sec / 1e9, "unit": "GCUPS", "cores": cores, "kind": "port",
            "sample": f"{n_sample} pairs of {length}x{length}, linear-space oracle port, {cores} threads", "seconds": sec}


def cpu_single_pair(a: np.ndarray, b: np.ndarray, p: int, what: str):
    """One pair through the reference's main_alignment_function (global + traceback), one host thread."""
    from oracle import pyoracle as po
    m, n = len(a), len(b)
    off = np.zeros(1, dtype=np.int64)
    la, lb = np.array([m], dtype=np.int32), np.array([n], dtype=np.int32)
    if po.have_ref():
        sec = po.ref_time_batch(np.ascontiguousarray(a), off, la, np.ascontiguousarray(b), off, lb, p, G, H, 1)
        return {"value": m * n / sec / 1e9, "unit": "GCUPS", "cores": 1, "kind": "reference", "seconds": sec,
                "sample": f"{what}: main_alignment_function(p={p}) on {m}x{n}, global + traceback, -O2, stdout to /dev/null"}
    t0 = time.perf_counter()
    po.score_linear(a.tobytes(), b.tobytes(), G, H, mode=po.GLOBAL)
    sec = time.perf_counter() - t0
    return {"value": m * n / sec / 1e9, "unit": "GCUPS", "cores": 1, "kind": "port", "seconds": sec,
            "sample": f"{what}: linear-space oracle port on {m}x{n}, score only"}


def run_reference(args, rank, world):
    """--impl reference: time the reference's own CPU path on this arm's config."""
    if rank != 0:
        return
    n = args.cpu_sample or 4096
    vals = []
    res = None
    for s in range(args.warmup + args.steps):
        res = cpu_baseline(n, 20250002 + s)
        if s >= args.warmup:
            vals.append(res)
    sec = float(np.mean([v["seconds"] for v in vals]))
    value = n * READ_LEN * READ_LEN / sec / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (exact integers)", "data": "synthetic",
            "config": dict(config_dict(args, world), pairs_per_step_sample=n),
            "cpu_baseline": {"value": value, "unit": "GCUPS", "cores": res["cores"], "kind": res["kind"],
                             "sample": res["sample"]},
            "e2e": {"value": value, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
def load_traffic_record():
    """DRAM bytes of the dominant kernel from a committed `ncu --set full` capture (profiles/r02_traffic.json names
    the kernel, the launch size and the commit it was captured on).  None when absent -- never a pasted constant."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    except Exception:
        return None


class Timer:
    """CUDA-event timing on the launch stream, barrier + synchronize on both sides, max over ranks."""

    def __init__(self, torch, dist, stream, dev, world):
        self.torch, self.dist, self.stream, self.dev, self.world = torch, dist, stream, dev, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, fn, steps, warmup):
        from cse305_parallel_sequence_alignment_b200 import sharding
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        ms = e0.elapsed_time(e1) / steps
        return sharding.max_over_ranks(ms, self.dev) if self.world > 1 else ms      # a rank-local timer must not enter a collective


DUMP_BYTES = 60_000_000     # the data of all files of one --dump-outputs run: under 64 MB with the .npy headers
DUMP_SEED = 20250010


def snapshot_outputs(torch, dItems, dOps, n, stride, world):
    """What the headline call hands back to its caller after a step: every pair's result record (psa_batch_item) and
    its traceback op words, copied to the host.  When all pairs do not fit in DUMP_BYTES, a seeded sample of them (the
    same on every run).  Returns (pair index, records [k, 10] int32, op words [k, stride] uint32)."""
    from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
    fields = len(ITEM_DTYPE.names)
    per_pair = 8 * (1 + fields + stride)
    k = min(n, DUMP_BYTES // world // per_pair)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
    sel = torch.from_numpy(idx).to(dItems.device)
    items = dItems.view(n, fields).index_select(0, sel).cpu().numpy()
    ops = dOps.view(n, stride).index_select(0, sel).cpu().numpy().view(np.uint32)
    return idx, items, ops


def write_outputs(path, snapshot, n, rank, world, dist):
    """DIR/<name>.npy as float64, which holds every int32 and uint32 exactly: one file per field of psa_batch_item,
    ops.npy ([pairs, stride] op words) and pair_index.npy (which pairs were kept).  With several ranks, rank 0 writes
    every rank's pairs, rank r's pair i as pair_index r * n + i."""
    from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
    idx, items, ops = snapshot
    if world > 1:
        parts = [None] * world if rank == 0 else None
        dist.gather_object((idx + rank * n, items, ops), parts, dst=0)
        if rank != 0:
            return
        idx, items, ops = (np.concatenate(x) for x in zip(*parts))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pair_index.npy"), idx.astype(np.float64))
    for c, name in enumerate(ITEM_DTYPE.names):
        np.save(os.path.join(path, f"{name}.npy"), items[:, c].astype(np.float64))
    np.save(os.path.join(path, "ops.npy"), ops.astype(np.float64))


def host_pack_record(psa, A, B):
    """CPU-only: ASCII reads -> the 2-bit fixed-stride layout on the host (psa_pack_reads, all host threads), i.e. what a
    caller holding ASCII reads pays per step before psa_align_batch_packed.  Never allowed to cost the headline."""
    try:
        outA = np.empty((A.shape[0], (A.shape[1] + 15) // 16), dtype=np.uint32)
        outB = np.empty((B.shape[0], (B.shape[1] + 15) // 16), dtype=np.uint32)
        outA.fill(0); outB.fill(0)              # a caller reuses its (page-locked) buffers: keep first-touch page faults out
        psa.pack_reads(A, 0, outA); psa.pack_reads(B, 0, outB)
        best = None
        for _ in range(12):                     # the minimum: the first calls after large allocations run several times slower
            t0 = time.perf_counter()
            _, bad_a = psa.pack_reads(A, 0, outA)
            _, bad_b = psa.pack_reads(B, 0, outB)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return {"ms_per_step": best * 1e3, "gbytes_per_s": (A.nbytes + B.nbytes) / best / 1e9, "threads": os.cpu_count() or 1,
                "non_acgt_bytes": int(bad_a + bad_b),
                "what": "psa_pack_reads on both sides of the step's reads (host only, outside every timed GPU region)"}
    except Exception as e:
        return {"error": repr(e)}


class LineEmitter:
    """Prints the ONE JSON line exactly once: on the normal path, or from a watchdog when the optional sub-records
    hang or fail on some rank (every rank then leaves with os._exit so that no collective is left waiting)."""

    def __init__(self, rank, line):
        self.rank, self.line, self.lock, self.done, self.timer = rank, line, threading.Lock(), False, None

    def _print(self, error=None):
        with self.lock:
            if self.done:
                return False
            self.done = True
            if self.rank == 0 and self.line is not None:
                if error is not None:
                    self.line["extra"] = {"error": error}
                print(json.dumps(self.line), flush=True)
            return True

    def arm(self, seconds, why):
        self.timer = threading.Timer(seconds, self.abort, args=(why,))
        self.timer.daemon = True
        self.timer.start()

    def abort(self, why):
        if self._print(why):
            sys.stdout.flush()
            os._exit(0)

    def finish(self):
        if self.timer:
            self.timer.cancel()
        self._print()


def extra_configs(args, psa, synth, torch, dist, ctx, T, rank, world, peak_s16, peak_s32, with_cpu):
    """Sub-records for BASELINE configs 1, 3, 4, 5 (SURVEY 8d)."""
    from cse305_parallel_sequence_alignment_b200 import multigpu, sharding
    from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
    dev, stream = T.dev, T.stream
    st = stream.cuda_stream
    out = {}

    def frac(cups, ops, pack, peak):
        return cups * ops / pack / peak

    # ---- config 1: the single gene_sequences_test pair (records #2 and #15, first 50 bp), global + traceback ----
    if rank == 0 and world == 1:
        from tests.helpers import dataset
        names, seqs = dataset()
        a, b = seqs[2][:50].encode(), seqs[15][:50].encode()
        for _ in range(3):
            ctx.align_pair(a, b, psa.GLOBAL, G, H)
        t0 = time.perf_counter()
        reps = 50
        for _ in range(reps):
            r = ctx.align_pair(a, b, psa.GLOBAL, G, H)
        sec = (time.perf_counter() - t0) / reps
        rec = {"workload": "config1: gene_sequences_test records #2 x #15, first 50 bp, global + traceback through psa_align_pair "
                           "(host buffers, synchronous)", "ms": sec * 1e3, "value": 2500 / sec / 1e9, "unit": "GCUPS",
               "corner": [r.t1, r.t2, r.t3], "bound": "launch + copy latency (2 500 cells)"}
        if with_cpu:
            av, bv = np.frombuffer(a, dtype=np.uint8), np.frombuffer(b, dtype=np.uint8)
            rec["cpu_baseline"] = cpu_single_pair(av, bv, 32, "the harness call as shipped")
        out["C1"] = rec

    # ---- config 3: 10 kbp x 10 kbp mutated copy, global, checkpointed traceback (replicas only: rank 0) ----
    if rank == 0:
        L = 10_000
        A, B = synth.mutated_pair(L, synth.SEED_C3)
        dA, dB = torch.from_numpy(A).to(dev), torch.from_numpy(B).to(dev)
        item = torch.zeros(10, dtype=torch.int32, device=dev)
        words = (2 * L + 15) // 16 + 1
        ops = torch.zeros(words, dtype=torch.int32, device=dev)

        def run3(tb):
            ctx.align_long_device(dA.data_ptr(), dB.data_ptr(), L, L, item.data_ptr(), ops.data_ptr() if tb else 0,
                                  words if tb else 0, psa.GLOBAL, G, H, tb, st)
        T1 = Timer(torch, dist, stream, dev, 1)
        ms_tb = T1.run(lambda: run3(True), 5, 2)
        ms_sc = T1.run(lambda: run3(False), 5, 2)
        run3(True)
        torch.cuda.synchronize()
        it = item.cpu().numpy().view(ITEM_DTYPE)[0]
        rec = {"workload": "config3: 10 kbp x 10 kbp mutated-copy pair, global alignment, checkpointed traceback (1 GPU; replicas only)",
               "ms": ms_tb, "value": L * L / ms_tb / 1e6, "unit": "GCUPS", "fill_only_ms": ms_sc, "aln_len": int(it["aln_len"]),
               "score": int(it["score"]),
               "roofline": {"bound": "latency (tile wavefront critical path: 118 dependent tile steps)", "unit": "Tlane-op/s",
                            "achieved": L * L / (ms_tb * 1e-3) * OPS_GLOBAL / 1e12, "peak": peak_s32 / 1e12,
                            "frac": frac(L * L / (ms_tb * 1e-3), OPS_GLOBAL, 1, peak_s32)}}
        if with_cpu and world == 1:
            rec["cpu_baseline"] = cpu_single_pair(A, B, 1, "the 10 kbp pair itself (2.4 GB of tables)")
        out["C3"] = rec

    # ---- config 4: ONE long pair, local score only; N GPUs = column strips streamed over NVLink ----
    L4 = args.c4_len
    A, B = synth.mutated_pair(L4, synth.SEED_C4)
    dA = torch.from_numpy(A).to(dev)
    item = torch.zeros(10, dtype=torch.int32, device=dev)
    if world == 1:
        dB = torch.from_numpy(B).to(dev)
        ms4 = T.run(lambda: ctx.align_long_device(dA.data_ptr(), dB.data_ptr(), L4, L4, item.data_ptr(), 0, 0, psa.LOCAL, G, H, False, st), 2, 1)
        it = item.cpu().numpy().view(ITEM_DTYPE)[0]
        res4 = (int(it["score"]), int(it["end_i"]), int(it["end_j"]))
    else:
        dB = torch.from_numpy(B).to(dev)
        pipe = multigpu.CyclicPanels(ctx, L4, rank, world)
        run4 = lambda: pipe.run(dA.data_ptr(), dB.data_ptr(), L4, L4, item.data_ptr(), psa.LOCAL, G, H, st)
        ms4 = T.run(run4, 2, 1)
        allit = sharding.gather_items(item.cpu().numpy().view(ITEM_DTYPE), [1] * world, dev)
        res4 = None
        if rank == 0:
            best = multigpu.merge_local_results(allit)
            res4 = (int(best["score"]), int(best["end_i"]), int(best["end_j"]))
        pipe.close()
    if rank == 0:
        cups4 = float(L4) * L4 / (ms4 * 1e-3)
        rec = {"workload": f"config4: {L4} x {L4} synthetic mutated-copy pair, local score + end cell, "
                           f"{'1 GPU' if world == 1 else f'block-cyclic systolic panels over {world} GPUs (NVLink peer stores)'}",
               "n_gpus": world, "scaling": "strong", "ms": ms4, "value": cups4 / 1e9, "unit": "GCUPS",
               "score": res4[0], "end": [res4[1], res4[2]],
               "roofline": {"bound": "int-alu", "unit": "Tlane-op/s", "achieved": cups4 * OPS_LOCAL / 1e12,
                            "peak": world * peak_s32 / 1e12, "frac": frac(cups4, OPS_LOCAL, 1, world * peak_s32), "pack": 1}}
        if with_cpu and world == 1:
            from oracle import pyoracle as po
            Lp = 20_000
            t0 = time.perf_counter()
            po.score_linear(A[:Lp].tobytes(), B[:Lp].tobytes(), G, H, mode=po.LOCAL)
            sec = time.perf_counter() - t0
            rec["cpu_baseline"] = {"value": Lp * Lp / sec / 1e9, "unit": "GCUPS", "cores": 1, "kind": "port", "seconds": sec,
                                   "sample": "20 kbp x 20 kbp prefix, local score, linear-space oracle port (the reference has no local "
                                             "mode and would need 24 TB of tables for the full pair)"}
        out["C4"] = rec
    del dA, dB

    # ---- config 5: 100 000 pairs of 5 kbp x 5 kbp, local score + end cell, sharded over the GPUs ----
    L5, total = 5000, args.c5_pairs
    lo, hi = sharding.shard_range(total, rank, world)
    n5 = hi - lo
    distinct = min(4096, n5)
    A5, B5 = synth.read_pair_batch(distinct, L5, synth.SEED_C5 + rank)
    reps5 = (n5 + distinct - 1) // distinct
    dA5 = torch.from_numpy(A5.reshape(-1)).to(dev).repeat(reps5)[:n5 * L5].contiguous()
    dB5 = torch.from_numpy(B5.reshape(-1)).to(dev).repeat(reps5)[:n5 * L5].contiguous()
    off5, len5 = synth.fixed_length_layout(n5, L5)
    dOff5, dLen5 = torch.from_numpy(off5).to(dev), torch.from_numpy(len5).to(dev)
    items5 = torch.zeros(n5 * 10, dtype=torch.int32, device=dev)
    ms5 = T.run(lambda: ctx.align_batch_device(dA5.data_ptr(), dOff5.data_ptr(), dLen5.data_ptr(), dB5.data_ptr(), dOff5.data_ptr(),
                                               dLen5.data_ptr(), n5, L5, L5, items5.data_ptr(), 0, 0, psa.LOCAL, G, H, False, st), 2, 1)
    if rank == 0:
        cups5 = float(total) * L5 * L5 / (ms5 * 1e-3)
        it5 = items5.cpu().numpy().view(ITEM_DTYPE)
        rec = {"workload": f"config5: {total} pairs of 5 kbp x 5 kbp (even: mutated copies, odd: random; {distinct} distinct pairs per "
                           f"rank tiled), local score + end cell, sharded over {world} GPU(s)",
               "n_gpus": world, "scaling": "strong", "ms": ms5, "value": cups5 / 1e9, "unit": "GCUPS",
               "mean_score_even": float(it5["score"][0::2].mean()), "mean_score_odd": float(it5["score"][1::2].mean()),
               "roofline": {"bound": "int-alu", "unit": "Tlane-op/s", "achieved": cups5 * OPS_LOCAL / 2 / 1e12,
                            "peak": world * peak_s16 / 1e12, "frac": frac(cups5, OPS_LOCAL, 2, world * peak_s16), "pack": 2}}
        if with_cpu and world == 1:
            cores = os.cpu_count() or 1
            rec["cpu_baseline"] = cpu_baseline(min(cores, 32), synth.SEED_C5, length=L5)
        out["C5"] = rec
    return out


# ------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import cse305_parallel_sequence_alignment_b200 as psa
    from cse305_parallel_sequence_alignment_b200 import synth, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = psa.Context(local_rank)

    # ---- this rank's shard, generated on the host into PINNED memory ----
    n = args.pairs
    A, B = synth.read_pair_batch(n, READ_LEN, synth.SEED_C2 + rank)
    off_np, len_np = synth.fixed_length_layout(n, READ_LEN)
    hA = torch.from_numpy(np.ascontiguousarray(A.reshape(-1))).pin_memory()
    hB = torch.from_numpy(np.ascontiguousarray(B.reshape(-1))).pin_memory()
    hOff = torch.from_numpy(off_np).pin_memory()
    hLen = torch.from_numpy(len_np).pin_memory()
    # the same reads as a production caller holds them: 2 bits per base, fixed stride (psa_align_batch_packed)
    hA2 = torch.from_numpy(psa.pack_reads_2bit(A).view(np.int32)).pin_memory()
    hB2 = torch.from_numpy(psa.pack_reads_2bit(B).view(np.int32)).pin_memory()
    stride = (2 * READ_LEN + 15) // 16 + 1
    hItems = torch.zeros(n * 10, dtype=torch.int32).pin_memory()
    hItems16 = torch.zeros(n * 4, dtype=torch.int32).pin_memory()
    hOps = torch.zeros(n * stride, dtype=torch.int32).pin_memory()
    items_np = hItems.numpy().view(psa.capi.ITEM_DTYPE)
    items16_np = hItems16.numpy().view(psa.capi.PACKED_ITEM_DTYPE)
    ops_np = hOps.numpy().view(np.uint32).reshape(n, stride)
    a2_np, b2_np = hA2.numpy().view(np.uint32), hB2.numpy().view(np.uint32)

    # ---- device-resident copy for the kernel-only measurement ----
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    dA, dB = hA.to(dev, non_blocking=True), hB.to(dev, non_blocking=True)
    dOff, dLen = hOff.to(dev, non_blocking=True), hLen.to(dev, non_blocking=True)
    dItems = torch.zeros(n * 10, dtype=torch.int32, device=dev)
    dOps = torch.zeros(n * stride, dtype=torch.int32, device=dev)
    cells_per_step = float(n) * READ_LEN * READ_LEN

    def step_device():
        ctx.align_batch_device(dA.data_ptr(), dOff.data_ptr(), dLen.data_ptr(), dB.data_ptr(), dOff.data_ptr(),
                               dLen.data_ptr(), n, READ_LEN, READ_LEN, dItems.data_ptr(), dOps.data_ptr(), stride,
                               psa.LOCAL, G, H, True, stream.cuda_stream)

    def step_e2e_packed():
        ctx.align_batch_packed(a2_np, b2_np, READ_LEN, READ_LEN, psa.LOCAL, G, H, True, items=items16_np, ops=ops_np, compact=True)

    def step_e2e_packed_fixed():
        ctx.align_batch_packed(a2_np, b2_np, READ_LEN, READ_LEN, psa.LOCAL, G, H, True, items=items16_np, ops=ops_np)

    def step_e2e_bytes():
        # every host array handed to the C-ABI lives in pinned memory (pageable offsets/lengths would turn the
        # library's asynchronous chunk copies into blocking staged ones)
        ctx.align_batch(hA.numpy(), hOff.numpy(), hLen.numpy(), hB.numpy(), hOff.numpy(), hLen.numpy(), psa.LOCAL, G, H,
                        True, items=items_np, ops=ops_np)

    T = Timer(torch, dist, stream, dev, world)

    def wall(fn, steps):
        for _ in range(2):
            fn()
        T.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        T.barrier()
        return sharding.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps, dev)

    # integer-issue peak, measured live (kind 1 = VIADDMNMX.S16x2, kind 0 = the int32 mix: the ALU pipe every DPX cell op runs on)
    peak_s16, _ = ctx.peak_int_ops(1)
    peak_s32, _ = ctx.peak_int_ops(0)

    warm = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    sampler.start()                      # runs through warm-up + timed steps: the GPU is under load throughout
    for _ in range(warm):
        step_device()
    T.barrier()
    launches0 = ctx.launches
    kernel_ms = T.run(step_device, args.steps, 0)
    launches = ctx.launches - launches0
    snapshot = None
    if args.dump_outputs:                # before the fill-only loop below overwrites the records
        snapshot = snapshot_outputs(torch, dItems, dOps, n, stride, world)

    # ---- the dominant kernel alone: same fill launches (direction codes included), walk kernels not launched ----
    ctx.set_option("pack_skip_walk", 1)      # measurement hook (csrc/psa_internal.h), not an environment switch
    l0 = ctx.launches
    fill_steps = max(3, args.steps // 2)
    fill_ms = T.run(step_device, fill_steps, 2)
    fill_launches_per_step = (ctx.launches - l0) // (fill_steps + 2) // 2     # one fill + one flagged-pair launch per chunk
    ctx.set_option("pack_skip_walk", 0)
    step_device()                        # leave complete results behind for the comparison below
    T.barrier()

    # ---- end to end through the host-buffer C-ABI (pinned host buffers, copies timed) ----
    e2e_ms = wall(step_e2e_packed, args.steps)
    same = bool(np.array_equal(dItems.cpu().numpy().view(psa.capi.ITEM_DTYPE)["score"], items16_np["score"]))
    e2e_fixed_ms = wall(step_e2e_packed_fixed, max(3, args.steps // 2))
    e2e_variants = None
    if args.e2e_variants:
        e2e_variants = []
        default_serial = 0
        for serial in (0, 1):
            ctx.set_option("pack_serial_fills", serial)
            for name, fn in (("fixed_stride_ops", step_e2e_packed_fixed), ("compact_ops", step_e2e_packed)):
                ms = wall(fn, max(3, args.steps // 2))
                e2e_variants.append({"serial_fills": serial, "ops": name, "ms_per_step": ms,
                                     "value": world * cells_per_step / (ms * 1e-3) / 1e9})
        ctx.set_option("pack_serial_fills", default_serial)
    e2e_bytes_ms = wall(step_e2e_bytes, max(3, args.steps // 2))
    clocks = sampler.stop()              # sampled while the GPU was busy (device-timed loop + e2e loops)
    if snapshot is not None:             # written once the clocks are no longer sampled
        write_outputs(args.dump_outputs, snapshot, n, rank, world, dist)
    same_bytes = bool(np.array_equal(items_np["score"], items16_np["score"]) and
                      np.array_equal(items_np["aln_len"].astype(np.int64), items16_np["aln_len"].astype(np.int64)))

    value = world * cells_per_step / (kernel_ms * 1e-3) / 1e9
    e2e_value = world * cells_per_step / (e2e_ms * 1e-3) / 1e9
    h2d = int(hA2.numel() * 4 + hB2.numel() * 4)
    # compact ops: only the words that carry ops come back (packed by the GPU straight into the pinned buffer)
    ops_words_back = int(psa.compact_ops_offsets(items16_np)[-1])
    d2h = int(hItems16.numel() * 4 + ops_words_back * 4)
    h2d_b = int(hA.numel() + hB.numel() + 2 * hOff.numel() * 8 + 2 * hLen.numel() * 4)
    d2h_b = int(hItems.numel() * 4 + hOps.numel() * 4)

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        per_gpu_cups = cells_per_step / (kernel_ms * 1e-3)
        PACK = 2                     # .S16x2: one lane-op updates two cells
        # roofline of the dominant kernel on ITS OWN duration (fill-only loop above); the whole-step view beside it
        fill_cups = cells_per_step / (fill_ms * 1e-3)
        achieved_lane = fill_cups * OPS_LOCAL / PACK
        step_lane = per_gpu_cups * OPS_LOCAL / PACK
        # dominant kernel = psa_pack_fill_kernel.  Algorithmic bytes per pair: both reads + offsets/lengths,
        # the 40 B result record, and the 5-bit direction codes it streams to the scratch ring
        # (ceil((150 + 7) / 4) blocks x 8 lanes x 128-byte lines for two pairs -> 20 480 B per pair).
        CODE_BYTES_PER_PAIR = ((READ_LEN + 7 + 3) // 4) * 8 * 128 // 2
        alg_bytes = n * (2 * READ_LEN + 2 * 8 + 2 * 4 + 40 + CODE_BYTES_PER_PAIR)
        pairs_per_launch = min(n, 131072)
        tr = load_traffic_record()
        traffic = None
        if tr and tr.get("kernel", "").startswith("psa_pack_fill_kernel") and tr.get("pairs_per_launch"):
            traffic = tr["dram_bytes_per_launch"] * pairs_per_launch / tr["pairs_per_launch"]
        roofline = {"bound": "int-alu", "achieved": achieved_lane / 1e12, "peak": peak_s16 / 1e12,
                    "unit": "Tlane-op/s", "frac": achieved_lane / peak_s16,
                    "traffic": traffic, "traffic_source": (tr or {}).get("source"),
                    "ops_per_cell": OPS_LOCAL, "pack": PACK,
                    "kernel": "psa_pack_fill_kernel<8,19,LOCAL,codes> (.S16x2 lanes, two pairs per register)",
                    "duration_basis": "fill launches alone (option pack_skip_walk, CUDA events on the launch stream, "
                                      "includes the ~1 % flagged-pair kernel)",
                    "kernel_ms_per_step": fill_ms, "launches_per_step": int(fill_launches_per_step),
                    "kernel_ms_per_launch": fill_ms / max(1, fill_launches_per_step),
                    "whole_step_frac": step_lane / peak_s16,
                    "peak_source": "psa_peak_int_ops(VIADDMNMX.S16x2) measured live in this run (ALU pipe, 64 lanes/clk/SM)",
                    "peak_tcups": peak_s16 * PACK / OPS_LOCAL / 1e12,
                    "int32_equivalent_frac": fill_cups * OPS_LOCAL / peak_s16,
                    "hbm": {"achieved": alg_bytes / (fill_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": alg_bytes / (fill_ms * 1e-3) / 1e9 / hbm_peak,
                            "algorithmic_bytes_per_launch": alg_bytes * pairs_per_launch / n,
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
        line = {"metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "s16x2", "data": "synthetic", "config": config_dict(args, world),
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms, "matches_device_pass": same,
                        "api": "psa_align_batch_packed + PSA_OPS_COMPACT (2-bit fixed-stride reads in pinned host memory -> 16-byte records + "
                               "2-bit op words back to back, written by the GPU straight into the pinned buffer as whole 128-byte lines)"},
                "e2e_fixed_stride_ops": {"value": world * cells_per_step / (e2e_fixed_ms * 1e-3) / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": h2d,
                                         "d2h_bytes_per_step": int(hItems16.numel() * 4 + hOps.numel() * 4), "ms_per_step": e2e_fixed_ms,
                                         "api": "psa_align_batch_packed without PSA_OPS_COMPACT (every pair's full 20-word op stride comes back)"},
                "e2e_variants": e2e_variants,
                "e2e_byte_api": {"value": world * cells_per_step / (e2e_bytes_ms * 1e-3) / 1e9, "unit": "GCUPS",
                                 "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b, "ms_per_step": e2e_bytes_ms,
                                 "matches_packed_api": same_bytes,
                                 "api": "psa_align_batch (raw bytes + offsets + lengths -> 40-byte records + 2-bit ops)"},
                "gpu_launches": int(launches), "roofline": roofline}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_sample or 20000, synth.SEED_C2, with_shipped=True)
            line["host_pack_2bit"] = host_pack_record(psa, A, B)

    del dA, dB, dOps, dItems
    emit = LineEmitter(rank, line)
    if not args.no_extra:
        # the headline must not be lost to a sub-record: a watchdog prints it (with the reason) and ends the process if
        # the sub-records raise on another rank or stall in a collective
        emit.arm(args.extra_timeout, "sub-records (configs 1/3/4/5) did not finish within %d s" % args.extra_timeout)
        try:
            extra = extra_configs(args, psa, synth, torch, dist, ctx, T, rank, world, peak_s16, peak_s32,
                                  with_cpu=(world == 1 and not args.no_cpu_baseline))
            if rank == 0:
                line["extra"] = {"configs": extra}
        except Exception as e:
            if world > 1:       # the other ranks may be waiting in a collective: print what we have and leave
                emit.abort(repr(e))
            if rank == 0:
                line["extra"] = {"error": repr(e)}
    emit.finish()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
