"""Batches of long pairs with traceback (config-5 shape, 5 kbp x 5 kbp) against the score-only batch and the per-pair
path, all device-resident, CUDA events after warm-up, at least MIN_SECONDS of work per figure.

    python tools/long_tb_bench.py [--pairs 4096] [--subset 64] [--out profiles/r03_long_tb.json]

Per mode (local, global):
  - tb_batch          psa_align_batch_device with PSA_WANT_TRACEBACK (checkpointed one-warp-per-pair fill + batched walk)
  - score_int32       the same call score only, int32 kernel (option pack = 0)
  - score_packed      the same call score only, default (packed .S16x2 kernel)
  - per_pair_subset   psa_align_long_device with traceback on the first --subset pairs, one after the other (each pair
                      over the whole GPU): measured on that subset only
  - fill / walk split of one tb_batch call from torch.profiler kernel times
  - check             tb_batch items and op words == per-pair items and op words, every pair of the batch
Sweep (local and global): 1, 2, 4, ... 64 pairs at 1 kbp and 5 kbp through both paths -- the pair-count threshold of the
host entry (psa_capi.cu, kLongTbBatchMin).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cse305_parallel_sequence_alignment_b200 as psa  # noqa: E402
from cse305_parallel_sequence_alignment_b200 import synth  # noqa: E402

MIN_SECONDS = 1.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power}


class Batch:
    """P pairs of L x L from the config-5 generator, resident on the device, with item / op buffers."""

    def __init__(self, P, L, seed=synth.SEED_C5):
        A, B = synth.read_pair_batch(P, L, seed)
        off, ln = synth.fixed_length_layout(P, L)
        self.P, self.L = P, L
        self.dA = torch.from_numpy(A.reshape(-1).copy()).cuda()
        self.dB = torch.from_numpy(B.reshape(-1).copy()).cuda()
        self.dOff, self.dLen = torch.from_numpy(off).cuda(), torch.from_numpy(ln).cuda()
        self.stride = (2 * L + 15) // 16 + 1
        self.items = torch.zeros(P * 10, dtype=torch.int32, device="cuda")
        self.ops = torch.zeros(P * self.stride, dtype=torch.int32, device="cuda")
        self.items_pp = torch.zeros(P * 10, dtype=torch.int32, device="cuda")
        self.ops_pp = torch.zeros(P * self.stride, dtype=torch.int32, device="cuda")
        self.cells = P * L * L

    def batch(self, ctx, mode, tb, stream, n=None):
        n = n or self.P
        ctx.align_batch_device(self.dA.data_ptr(), self.dOff.data_ptr(), self.dLen.data_ptr(), self.dB.data_ptr(),
                               self.dOff.data_ptr(), self.dLen.data_ptr(), n, self.L, self.L, self.items.data_ptr(),
                               self.ops.data_ptr() if tb else 0, self.stride if tb else 0, mode, 1, 2, tb, stream.cuda_stream)

    def per_pair(self, ctx, mode, stream, n):
        for k in range(n):
            ctx.align_long_device(self.dA.data_ptr() + k * self.L, self.dB.data_ptr() + k * self.L, self.L, self.L,
                                  self.items_pp.data_ptr() + 40 * k, self.ops_pp.data_ptr() + 4 * k * self.stride,
                                  self.stride, mode, 1, 2, True, stream.cuda_stream)


def timed(fn, stream):
    """ms per call: one warm-up call, then repeats until MIN_SECONDS of events-timed work."""
    fn()
    torch.cuda.synchronize()
    reps, total = 0, 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while total < MIN_SECONDS * 1e3:
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        total += e0.elapsed_time(e1)
        reps += 1
    return total / reps, reps


def fill_walk_split(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"fill_ms": 0.0, "walk_ms": 0.0}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if "batch_tb_fill" in ev.key:
            out["fill_ms"] += us / 1e3
        elif "batch_tb_walk" in ev.key:
            out["walk_ms"] += us / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--len", type=int, default=5000)
    ap.add_argument("--subset", type=int, default=64)
    ap.add_argument("--sweep", default="1000,5000")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_long_tb.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_tb_bench.py needs a CUDA device")
    rec = {"card": card(), "shape": f"{args.pairs} x {args.len} x {args.len}, synth.read_pair_batch(SEED_C5), g=1 h=2",
           "min_seconds_per_figure": MIN_SECONDS, "modes": {}, "sweep": []}
    ctx = psa.Context(0)
    int32 = psa.Context(0)
    int32.set_option("pack", 0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    big = Batch(args.pairs, args.len)
    for mode, name in ((psa.LOCAL, "local"), (psa.GLOBAL, "global")):
        r = {}
        for key, c, tb in (("tb_batch", ctx, True), ("score_int32", int32, False), ("score_packed", ctx, False)):
            ms, reps = timed(lambda: big.batch(c, mode, tb, stream), stream)
            r[key] = {"ms": round(ms, 3), "reps": reps, "gcups": round(big.cells / ms / 1e6, 1)}
        sub = min(args.subset, args.pairs)
        ms, reps = timed(lambda: big.per_pair(ctx, mode, stream, sub), stream)
        r["per_pair_subset"] = {"pairs": sub, "ms": round(ms, 3), "reps": reps,
                                "gcups": round(sub * args.len * args.len / ms / 1e6, 1)}
        r["tb_over_score_int32"] = round(r["tb_batch"]["ms"] / r["score_int32"]["ms"], 3)
        r["split"] = {k: round(v, 3) for k, v in fill_walk_split(lambda: big.batch(ctx, mode, True, stream)).items()}
        # byte-identical check: every pair of the batch against the per-pair path
        big.batch(ctx, mode, True, stream)
        big.per_pair(ctx, mode, stream, args.pairs)
        torch.cuda.synchronize()
        same_items = bool(torch.equal(big.items, big.items_pp))
        same_ops = bool(torch.equal(big.ops, big.ops_pp))
        r["check"] = {"pairs": args.pairs, "items_identical": same_items, "ops_identical": same_ops}
        rec["modes"][name] = r
        print(name, json.dumps(r), flush=True)
    del big
    torch.cuda.empty_cache()
    for L in [int(x) for x in args.sweep.split(",")]:
        sw = Batch(64, L, seed=synth.SEED_C5 + L)
        for mode, name in ((psa.LOCAL, "local"), (psa.GLOBAL, "global")):
            n = 1
            while n <= 64:
                tb_ms, _ = timed(lambda: sw.batch(ctx, mode, True, stream, n), stream)
                pp_ms, _ = timed(lambda: sw.per_pair(ctx, mode, stream, n), stream)
                row = {"len": L, "mode": name, "pairs": n, "batch_ms": round(tb_ms, 3), "per_pair_ms": round(pp_ms, 3),
                       "per_pair_over_batch": round(pp_ms / tb_ms, 3)}
                rec["sweep"].append(row)
                print(json.dumps(row), flush=True)
                n *= 2
        del sw
    rec["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
