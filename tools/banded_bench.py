"""Banded batches (psa_align_batch_banded_device) on the config-5 shape, against the unbanded traceback batch and the
int32 and packed score-only batches on the same pairs; device-resident, CUDA events after warm-up, at least
MIN_SECONDS of work per figure.

    python tools/banded_bench.py [--pairs 4096] [--len 5000] [--bands 64,128,256,512] [--out profiles/r04_banded.json]

Per mode (local, global):
  - tb_batch / score_int32 / score_packed     the unbanded psa_align_batch_device calls (as tools/long_tb_bench.py)
  - banded[band].tb / banded[band].score      psa_align_batch_banded_device with / without PSA_WANT_TRACEBACK
  - banded[band].same_as_unbanded_even        of the even pairs (B a mutated copy of A), how many banded traceback
                                              records and op words equal the unbanded ones
  - banded[band].score_equals_tb              score-only items == traceback items on every field both report
One 1 Mbp pair (synth.mutated_pair(1e6, SEED_C4)), band 1000, global, traceback: time of one call and the device memory
the context allocated for it.
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
from long_tb_bench import MIN_SECONDS, Batch, card, timed  # noqa: E402

FIELDS = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j")


def banded(ctx, bt, band, mode, tb, stream, items, ops):
    ctx.align_batch_banded_device(bt.dA.data_ptr(), bt.dOff.data_ptr(), bt.dLen.data_ptr(), bt.dB.data_ptr(), bt.dOff.data_ptr(),
                                  bt.dLen.data_ptr(), bt.P, bt.L, bt.L, band, items.data_ptr(), ops.data_ptr() if tb else 0,
                                  bt.stride if tb else 0, mode, 1, 2, tb, stream.cuda_stream)


def one_mbp(band):
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    dA, dB = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    off, ln = torch.zeros(1, dtype=torch.int64, device="cuda"), torch.full((1,), len(A), dtype=torch.int32, device="cuda")
    stride = (2 * len(A) + 15) // 16 + 1
    items = torch.zeros(10, dtype=torch.int32, device="cuda")
    ops = torch.zeros(stride, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    ctx = psa.Context(0)
    stream = torch.cuda.Stream()

    def call():
        ctx.align_batch_banded_device(dA.data_ptr(), off.data_ptr(), ln.data_ptr(), dB.data_ptr(), off.data_ptr(), ln.data_ptr(),
                                      1, len(A), len(B), band, items.data_ptr(), ops.data_ptr(), stride, psa.GLOBAL, 1, 2, True,
                                      stream.cuda_stream)
    ms, reps = timed(call, stream)
    free1, _ = torch.cuda.mem_get_info()
    it = items.cpu().numpy().view(psa.capi.ITEM_DTYPE)[0]
    ctx.close()
    return {"shape": "1 Mbp x 1 Mbp, synth.mutated_pair(SEED_C4), global, g=1 h=2", "band": band, "ms": round(ms, 3),
            "reps": reps, "context_allocated_GiB": round((free0 - free1) / 2**30, 3), "score": int(it["score"]),
            "aln_len": int(it["aln_len"])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--len", type=int, default=5000)
    ap.add_argument("--bands", default="64,128,256,512")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_banded.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("banded_bench.py needs a CUDA device")
    rec = {"card": card(), "shape": f"{args.pairs} x {args.len} x {args.len}, synth.read_pair_batch(SEED_C5), g=1 h=2",
           "min_seconds_per_figure": MIN_SECONDS, "modes": {}}
    ctx = psa.Context(0)
    int32 = psa.Context(0)
    int32.set_option("pack", 0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    bt = Batch(args.pairs, args.len)
    b_items = torch.zeros_like(bt.items)
    b_ops = torch.zeros_like(bt.ops)
    s_items = torch.zeros_like(bt.items)
    even = np.arange(0, args.pairs, 2)
    for mode, name in ((psa.LOCAL, "local"), (psa.GLOBAL, "global")):
        r = {}
        for key, c, tb in (("tb_batch", ctx, True), ("score_int32", int32, False), ("score_packed", ctx, False)):
            ms, reps = timed(lambda: bt.batch(c, mode, tb, stream), stream)
            r[key] = {"ms": round(ms, 3), "reps": reps}
        bt.batch(ctx, mode, True, stream)
        torch.cuda.synchronize()
        ref_items = bt.items.cpu().numpy().view(psa.capi.ITEM_DTYPE).copy()
        ref_ops = bt.ops.cpu().numpy().reshape(args.pairs, bt.stride).copy()
        r["banded"] = {}
        for band in [int(x) for x in args.bands.split(",")]:
            tb_ms, tb_reps = timed(lambda: banded(ctx, bt, band, mode, True, stream, b_items, b_ops), stream)
            sc_ms, sc_reps = timed(lambda: banded(ctx, bt, band, mode, False, stream, s_items, b_ops), stream)
            torch.cuda.synchronize()
            items = b_items.cpu().numpy().view(psa.capi.ITEM_DTYPE).copy()
            ops = b_ops.cpu().numpy().reshape(args.pairs, bt.stride).copy()
            sitems = s_items.cpu().numpy().view(psa.capi.ITEM_DTYPE)
            same = 0
            for k in even:
                L = (int(items[k]["aln_len"]) + 15) // 16
                same += int(items[k].tobytes() == ref_items[k].tobytes() and np.array_equal(ops[k, :L], ref_ops[k, :L]))
            row = {"tb_ms": round(tb_ms, 3), "tb_reps": tb_reps, "score_ms": round(sc_ms, 3), "score_reps": sc_reps,
                   "tb_speedup_vs_unbanded_tb": round(r["tb_batch"]["ms"] / tb_ms, 2),
                   "score_speedup_vs_packed": round(r["score_packed"]["ms"] / sc_ms, 2),
                   "score_speedup_vs_int32": round(r["score_int32"]["ms"] / sc_ms, 2),
                   "same_as_unbanded_even": f"{same}/{len(even)}",
                   "score_equals_tb": bool(all(np.array_equal(sitems[f], items[f]) for f in FIELDS))}
            r["banded"][band] = row
            print(name, band, json.dumps(row), flush=True)
        rec["modes"][name] = r
        print(name, json.dumps({k: v for k, v in r.items() if k != "banded"}), flush=True)
    del bt
    ctx.close()
    int32.close()
    torch.cuda.empty_cache()
    rec["one_mbp"] = one_mbp(1000)
    print(json.dumps(rec["one_mbp"]), flush=True)
    rec["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
