"""One banded pair over the whole GPU (psa_align_long_banded_device) against the one-warp path (a one-pair
psa_align_batch_banded_device) on the C4 pair, synth.mutated_pair(1e6, SEED_C4); device-resident, CUDA events after a
warm-up, at least MIN_SECONDS of work per figure (one-warp figures that take longer than that: one call after the
warm-up of the same kernels at a narrower band).

    python tools/banded_pair_bench.py [--bands 100,1000,10000,100000,1000000] [--out profiles/r05_banded_pair.json]

Per mode (global, local) and band:
  - pair.score_ms / pair.tb_ms              the new entry, each timed twice (the spread of two runs)
  - one_warp.score_ms / one_warp.tb_ms      the one-warp path, where it takes <= ONE_WARP_MAX_S (else "not run")
  - same_as_one_warp                        records and op words of both paths equal, where both ran
  - context_allocated_MiB                   device memory a fresh context allocated for the new entry's calls
Traceback runs where the checkpoints fit; band 1000000 (>= max(m, n), every cell) is the score-only grid's other side.
Also: the unbanded psa_align_long_device score-only time, and the fill / tile-offset / code-recompute / walk split of
one traceback call at band 1000 from torch.profiler (a separate call after the timed ones).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import cse305_parallel_sequence_alignment_b200 as psa  # noqa: E402
from cse305_parallel_sequence_alignment_b200 import synth  # noqa: E402
from long_tb_bench import MIN_SECONDS, card, timed  # noqa: E402

ONE_WARP_MAX_S = 30.0
ONE_WARP_CELLS_PER_S = 0.7e9          # one warp, traceback fill (profiles/r04_banded.json): only decides what to run


class Pair:
    def __init__(self, A, B):
        self.m, self.n = len(A), len(B)
        self.dA, self.dB = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
        self.off = torch.zeros(1, dtype=torch.int64, device="cuda")
        self.la = torch.full((1,), self.m, dtype=torch.int32, device="cuda")
        self.lb = torch.full((1,), self.n, dtype=torch.int32, device="cuda")
        self.words = (self.m + self.n + 15) // 16 + 1
        self.items = torch.zeros(10, dtype=torch.int32, device="cuda")
        self.ops = torch.zeros(self.words, dtype=torch.int32, device="cuda")

    def pair(self, ctx, band, mode, tb, stream):
        ctx.align_long_banded_device(self.dA.data_ptr(), self.dB.data_ptr(), self.m, self.n, band, self.items.data_ptr(),
                                     self.ops.data_ptr() if tb else 0, self.words if tb else 0, mode, 1, 2, tb,
                                     stream.cuda_stream)

    def one_warp(self, ctx, band, mode, tb, stream):
        ctx.align_batch_banded_device(self.dA.data_ptr(), self.off.data_ptr(), self.la.data_ptr(), self.dB.data_ptr(),
                                      self.off.data_ptr(), self.lb.data_ptr(), 1, self.m, self.n, band, self.items.data_ptr(),
                                      self.ops.data_ptr() if tb else 0, self.words if tb else 0, mode, 1, 2, tb,
                                      stream.cuda_stream)

    def result(self):
        it = self.items.cpu().numpy().view(psa.capi.ITEM_DTYPE)[0].copy()
        L = (int(it["aln_len"]) + 15) // 16
        return it, self.ops.cpu().numpy()[:L].copy()


def once(fn, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bands", default="100,1000,10000,100000,1000000")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_banded_pair.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("banded_pair_bench.py needs a CUDA device")
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    P = Pair(A, B)
    stream = torch.cuda.Stream()
    rec = {"card": card(), "shape": "1 Mbp x 1 Mbp, synth.mutated_pair(SEED_C4), g=1 h=2",
           "min_seconds_per_figure": MIN_SECONDS, "one_warp_max_seconds": ONE_WARP_MAX_S, "modes": {}}
    ctx = psa.Context(0)
    for mode, name in ((psa.GLOBAL, "global"), (psa.LOCAL, "local")):
        r = {}
        ms, reps = timed(lambda: ctx.align_long_device(P.dA.data_ptr(), P.dB.data_ptr(), P.m, P.n, P.items.data_ptr(),
                                                       mode=mode, traceback=False, stream=stream.cuda_stream), stream)
        r["unbanded_long_device_score"] = {"ms": round(ms, 3), "reps": reps}
        r["bands"] = {}
        for band in [int(x) for x in args.bands.split(",")]:
            row = {}
            torch.cuda.synchronize()
            free0, _ = torch.cuda.mem_get_info()
            c = psa.Context(0)
            for tb in (False, True):
                key = "tb" if tb else "score"
                if tb and band >= max(P.m, P.n):
                    row[key] = "not run: the checkpoints of every cell do not fit"
                    continue
                try:
                    a = timed(lambda: P.pair(c, band, mode, tb, stream), stream)
                    b = timed(lambda: P.pair(c, band, mode, tb, stream), stream)
                except psa.PsaError as e:
                    row[key] = f"not run: {e}"
                    continue
                got = P.result()
                row[key] = {"ms": [round(a[0], 3), round(b[0], 3)], "reps": [a[1], b[1]], "launches_per_call": None}
                n0 = c.launches
                P.pair(c, band, mode, tb, stream)
                row[key]["launches_per_call"] = c.launches - n0
                est = P.m * (2.0 * min(band, P.n) + 1) / ONE_WARP_CELLS_PER_S
                if est > ONE_WARP_MAX_S:
                    row[key]["one_warp"] = f"not run (estimated {est:.0f} s)"
                    continue
                if est * 1e3 > 2 * MIN_SECONDS * 1e3:
                    ow, owr = once(lambda: P.one_warp(ctx, band, mode, tb, stream), stream), 1
                else:
                    ow, owr = timed(lambda: P.one_warp(ctx, band, mode, tb, stream), stream)
                want = P.result()
                row[key]["one_warp"] = {"ms": round(ow, 3), "reps": owr}
                row[key]["speedup_vs_one_warp"] = round(ow / max(a[0], b[0]), 2)
                row[key]["same_as_one_warp"] = bool(got[0].tobytes() == want[0].tobytes() and np.array_equal(got[1], want[1]))
                print(name, band, key, json.dumps(row[key]), flush=True)
            torch.cuda.synchronize()
            free1, _ = torch.cuda.mem_get_info()
            c.close()
            row["context_allocated_MiB"] = round((free0 - free1) / 2**20, 1)
            r["bands"][band] = row
            print(name, band, json.dumps(row), flush=True)
        rec["modes"][name] = r
    # fill / tile offsets / code recompute / walk of one traceback call, from the profiler in a call of its own
    split = {}
    for band in (1000, 10000):
        P.pair(ctx, band, psa.GLOBAL, True, stream)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            P.pair(ctx, band, psa.GLOBAL, True, stream)
            torch.cuda.synchronize()
        parts = {}
        for ev in prof.key_averages():
            for k in ("psa_banded_pair_fill_kernel", "psa_banded_tile_base_kernel", "psa_banded_pair_codes_kernel",
                      "psa_banded_pair_walk_kernel"):
                if k in ev.key:
                    parts[k] = parts.get(k, 0.0) + ev.device_time_total / 1e3
        split[band] = {k: round(v, 3) for k, v in parts.items()}
        print("split", band, json.dumps(split[band]), flush=True)
    rec["split_global_tb_ms"] = split
    ctx.close()
    rec["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
