"""Banded alignment along an anchor chain (psa_align_batch_guided_device, psa_align_pair_guided): what the chain costs
and what it buys.  Device-resident batches, CUDA events after a warm-up, at least MIN_SECONDS of work per figure; the
card's name and power limit are read in the same run.

    python tools/guided_bench.py [--pairs 4096] [--len 5000] [--bands 64,128,256,512] [--out profiles/r06_guided.json]

overhead (4096 x 5 kbp pairs of config 5, both modes, traceback and score only, per band):
  banded        psa_align_batch_banded_device
  empty         psa_align_batch_guided_device with empty chains       (records must equal banded's)
  diag16        the same with 16 anchors on the diagonal of every pair  (records must equal empty's)
payoff:
  sv            512 x 5 kbp pairs with one 500 - 2000 bp insertion in A or B, chains at the breakpoints, global
                traceback: guided band 64 against the smallest plain band that reaches the same scores and against
                the unbanded traceback batch
  one_mbp       the 1 Mbp C4 pair with a 10 kbp insertion in A and one in B: psa_align_pair_guided at band 100 against
                psa_align_pair_banded at bands up to the one that reaches the same score, and psa_align_long_device
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
from tests.helpers import mutated_copy, random_dna  # noqa: E402

ITEM = psa.capi.ITEM_DTYPE


def dev_anchors(chains):
    anc, off, cnt = psa.pack_anchors(chains)
    return (torch.from_numpy(np.concatenate([anc.reshape(-1), np.zeros(2, np.int32)])).cuda(), torch.from_numpy(off).cuda(),
            torch.from_numpy(cnt).cuda())


class Run:
    def __init__(self, ctx, bt, stream):
        self.ctx, self.bt, self.stream = ctx, bt, stream
        self.items = torch.zeros_like(bt.items)
        self.ops = torch.zeros_like(bt.ops)

    def banded(self, band, mode, tb):
        bt = self.bt
        self.ctx.align_batch_banded_device(bt.dA.data_ptr(), bt.dOff.data_ptr(), bt.dLen.data_ptr(), bt.dB.data_ptr(),
                                           bt.dOff.data_ptr(), bt.dLen.data_ptr(), bt.P, bt.L, bt.L, band, self.items.data_ptr(),
                                           self.ops.data_ptr() if tb else 0, bt.stride if tb else 0, mode, 1, 2, tb,
                                           self.stream.cuda_stream)

    def guided(self, anc, band, mode, tb):
        bt = self.bt
        self.ctx.align_batch_guided_device(bt.dA.data_ptr(), bt.dOff.data_ptr(), bt.dLen.data_ptr(), bt.dB.data_ptr(),
                                           bt.dOff.data_ptr(), bt.dLen.data_ptr(), bt.P, bt.L, bt.L, anc[0].data_ptr(),
                                           anc[1].data_ptr(), anc[2].data_ptr(), band, self.items.data_ptr(),
                                           self.ops.data_ptr() if tb else 0, bt.stride if tb else 0, mode, 1, 2, tb,
                                           self.stream.cuda_stream)

    def result(self):
        torch.cuda.synchronize()
        return self.items.cpu().numpy().tobytes() + self.ops.cpu().numpy().tobytes()


def overhead(args, stream):
    ctx = psa.Context(0)
    bt = Batch(args.pairs, args.len)
    run = Run(ctx, bt, stream)
    L = args.len
    empty = dev_anchors([[]] * bt.P)
    diag = dev_anchors([[[k * L // 17, k * L // 17] for k in range(1, 17)]] * bt.P)
    out = {}
    for mode, name in ((psa.LOCAL, "local"), (psa.GLOBAL, "global")):
        out[name] = {}
        for band in [int(x) for x in args.bands.split(",")]:
            row = {}
            for tb, kind in ((True, "tb"), (False, "score")):
                ms_b, _ = timed(lambda: run.banded(band, mode, tb), stream)
                ref = run.result()
                ms_e, _ = timed(lambda: run.guided(empty, band, mode, tb), stream)
                same_e = run.result() == ref
                ms_d, _ = timed(lambda: run.guided(diag, band, mode, tb), stream)
                same_d = run.result() == ref
                row[kind] = {"banded_ms": round(ms_b, 3), "empty_ms": round(ms_e, 3), "diag16_ms": round(ms_d, 3),
                             "empty_over_banded": round(ms_e / ms_b, 4), "diag16_over_empty": round(ms_d / ms_e, 4),
                             "empty_equals_banded": same_e, "diag16_equals_banded": same_d}
            out[name][band] = row
            print("overhead", name, band, json.dumps(row), flush=True)
    ctx.close()
    return out


def sv_pair(seed, L=5000):
    """tests/test_gpu_guided.py's structural-variant pair: one 500 - 2000 bp insertion, 3 % substitutions."""
    rng = np.random.default_rng(seed)
    x = random_dna(rng, L)
    y = mutated_copy(rng, x, L, sub=0.03, ins=0.0, dele=0.0)
    n_ins, p = int(rng.integers(500, 2001)), int(rng.integers(1000, 4000))
    ins = random_dna(rng, n_ins)
    if seed % 2 == 0:
        return x[:p] + ins + x[p:], y, [[p, p], [p + n_ins, p]]
    return x, y[:p] + ins + y[p:], [[p, p], [p, p + n_ins]]


def sv_payoff(stream, n_pairs=512):
    As, Bs, chains = zip(*[sv_pair(20000 + k) for k in range(n_pairs)])
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    M, N = int(la.max()), int(lb.max())
    d = [torch.from_numpy(x).cuda() for x in (np.concatenate([ba, [0]]).astype(np.uint8), oa, la,
                                              np.concatenate([bb, [0]]).astype(np.uint8), ob, lb)]
    anc = dev_anchors(chains)
    stride = (M + N + 15) // 16 + 1
    items = torch.zeros(n_pairs * 10, dtype=torch.int32, device="cuda")
    ops = torch.zeros(n_pairs * stride, dtype=torch.int32, device="cuda")
    ctx = psa.Context(0)
    args = (d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(), n_pairs, M, N)

    def scores():
        torch.cuda.synchronize()
        return items.cpu().numpy().view(ITEM)["score"].copy()

    out = {"shape": f"{n_pairs} pairs, 5 kbp + one 500 - 2000 bp insertion in A or B, 3 % substitutions, global traceback"}
    ms, reps = timed(lambda: ctx.align_batch_device(*args, items.data_ptr(), ops.data_ptr(), stride, psa.GLOBAL, 1, 2, True,
                                                    stream.cuda_stream), stream)
    full = scores()
    out["unbanded_tb_ms"] = round(ms, 3)
    ms, reps = timed(lambda: ctx.align_batch_guided_device(*args, anc[0].data_ptr(), anc[1].data_ptr(), anc[2].data_ptr(), 64,
                                                           items.data_ptr(), ops.data_ptr(), stride, psa.GLOBAL, 1, 2, True,
                                                           stream.cuda_stream), stream)
    g = scores()
    out["guided64_tb_ms"] = round(ms, 3)
    out["guided64_reaches_unbanded"] = f"{int((g == full).sum())}/{n_pairs}"
    out["plain"] = {}
    for band in (64, 256, 1024, 2048, 4096):
        ms, reps = timed(lambda: ctx.align_batch_banded_device(*args, band, items.data_ptr(), ops.data_ptr(), stride, psa.GLOBAL,
                                                               1, 2, True, stream.cuda_stream), stream)
        s = scores()
        out["plain"][band] = {"tb_ms": round(ms, 3), "reaches_unbanded": f"{int((s == full).sum())}/{n_pairs}"}
        print("sv plain", band, json.dumps(out["plain"][band]), flush=True)
        if (s == full).all():
            break
    print("sv", json.dumps({k: v for k, v in out.items() if k != "plain"}), flush=True)
    ctx.close()
    return out


def one_mbp_payoff():
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    rng = np.random.default_rng(9600)
    a = A[:300_000].tobytes() + random_dna(rng, 10_000) + A[300_000:].tobytes()
    b = B[:700_000].tobytes() + random_dna(rng, 10_000) + B[700_000:].tobytes()
    chain = [[300_000, 300_000], [310_000, 300_000], [710_000, 700_000], [710_000, 710_000]]
    ctx = psa.Context(0)
    out = {"shape": "1 Mbp C4 pair + 10 kbp insertion in A at 300 kbp and in B at 700 kbp, global traceback, host strings"}

    def clock(fn):
        fn()                                               # warm-up: allocations and module loading
        t0 = time.perf_counter()
        r = fn()
        return r, (time.perf_counter() - t0) * 1e3

    r, ms = clock(lambda: ctx.align_pair_guided(a, b, chain, 100))
    out["guided100"] = {"ms": round(ms, 1), "score": r.score}
    out["plain"] = {}
    for band in (100, 1000, 10_000, 20_000):
        rp, ms = clock(lambda: ctx.align_pair_banded(a, b, band))
        out["plain"][band] = {"ms": round(ms, 1), "score": rp.score}
        print("1Mbp plain", band, out["plain"][band], flush=True)
        if rp.score >= r.score:
            break
    dA = torch.frombuffer(bytearray(a), dtype=torch.uint8).cuda()
    dB = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
    words = (len(a) + len(b) + 15) // 16 + 1
    item = torch.zeros(10, dtype=torch.int32, device="cuda")
    ops = torch.zeros(words, dtype=torch.int32, device="cuda")

    def unbanded():
        ctx.align_long_device(dA.data_ptr(), dB.data_ptr(), len(a), len(b), item.data_ptr(), ops.data_ptr(), words,
                              psa.GLOBAL, 1, 2, True)
        torch.cuda.synchronize()
        return int(item[3])
    s, ms = clock(unbanded)
    out["unbanded_long_device"] = {"ms": round(ms, 1), "score": s}
    print("1Mbp", json.dumps(out), flush=True)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--len", type=int, default=5000)
    ap.add_argument("--bands", default="64,128,256,512")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_guided.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("guided_bench.py needs a CUDA device")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    rec = {"card": card(), "overhead_shape": f"{args.pairs} x {args.len} x {args.len}, synth.read_pair_batch(SEED_C5), g=1 h=2",
           "min_seconds_per_figure": MIN_SECONDS}
    rec["overhead"] = overhead(args, stream)
    torch.cuda.empty_cache()
    rec["sv"] = sv_payoff(stream)
    torch.cuda.empty_cache()
    rec["one_mbp"] = one_mbp_payoff()
    rec["measured_at"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
