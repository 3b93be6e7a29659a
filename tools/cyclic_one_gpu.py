"""The multi-rank data path of config 4 on ONE GPU: W "ranks" = W contexts with their own streams in one process,
each running its block-cyclic share of the panels through psa_align_long_cyclic_device, the inter-rank rings being
ordinary device buffers of the same GPU (rank r's outgoing ring = rank (r+1) mod W's incoming buffer, no CUDA IPC,
no NVLink).  Everything else is what N GPUs run: in-band lap tags, cumulative row numbering over back-to-back calls,
the consumed-rows back-pressure, has_in / has_out panels, the per-rank best that the host merges.  The result must
equal the CPU oracle.  Used by tests/test_multigpu.py so that a 1-GPU box exercises the rings too.

Env: M, N (lengths), CALLS, and either WORLD, PANEL_STRIPS, KC (columns per lane: 8 or 4), MODE (1 local / 0 global) or
VARIANTS = JSON list of {"world":, "panel_strips":, "kc":, "mode":} run one after the other (one JSON line each).  A variant
may add "unaligned_rank": r and "a_offset": 1-3: rank r then reads A at that byte offset from a 4-byte boundary, which
runs its panels with 2-row steps while the other ranks take 4-row steps."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cse305_parallel_sequence_alignment_b200 as psa  # noqa: E402
from cse305_parallel_sequence_alignment_b200 import multigpu, synth  # noqa: E402
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE  # noqa: E402
from oracle import pyoracle as po  # noqa: E402  (the checker)


def main():
    m, n = int(os.environ.get("M", "12000")), int(os.environ.get("N", "20000"))
    calls = int(os.environ.get("CALLS", "2"))
    variants = json.loads(os.environ.get("VARIANTS", "null")) or [
        {"world": int(os.environ.get("WORLD", "2")), "panel_strips": int(os.environ.get("PANEL_STRIPS", "8")),
         "kc": int(os.environ.get("KC", "8")), "mode": int(os.environ.get("MODE", str(psa.LOCAL)))}]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    A, B = synth.mutated_pair(max(m, n), synth.SEED_C4)
    A, B = np.ascontiguousarray(A[:m]), np.ascontiguousarray(B[:n])
    dA, dB = torch.from_numpy(A).to(dev), torch.from_numpy(B).to(dev)
    oracle = {}
    for v in variants:
        mode = int(v.get("mode", psa.LOCAL))
        if mode not in oracle:
            oracle[mode] = po.score_linear(A.tobytes(), B.tobytes(), 1, 2, mode=mode)
        one_variant(dev, A, B, dA, dB, m, n, int(v.get("world", 2)), int(v.get("panel_strips", 8)), int(v.get("kc", 8)), mode, calls,
                    oracle[mode], int(v.get("unaligned_rank", -1)), int(v.get("a_offset", 0)))


def one_variant(dev, A, B, dA, dB, m, n, world, ps, kc, mode, calls, lin, unaligned_rank=-1, a_offset=0):
    ctxs, streams, items, xin = [], [], [], []
    a_ptr = [dA.data_ptr()] * world
    if 0 <= unaligned_rank < world and a_offset % 4:
        shifted = torch.zeros(m + 4, dtype=torch.uint8, device=dev)
        shifted[a_offset:a_offset + m] = dA
        a_ptr[unaligned_rank] = shifted.data_ptr() + a_offset
    for r in range(world):
        c = psa.Context(0)
        c.set_option("systolic_kc", kc)
        ctxs.append(c)
        streams.append(torch.cuda.Stream(device=dev))
        items.append(torch.zeros(10, dtype=torch.int32, device=dev))
        xin.append(c.xbuf_create(m)[0])
    cols = ctxs[0].long_strip_columns
    # the kernel state of every context is allocated by one single-rank call first: a first-use allocation in the
    # middle of the W-rank launch would synchronise the device while rank 0's later panels wait for ranks not launched yet
    for r in range(world):
        ctxs[r].align_long_cyclic_device(a_ptr[r], dB.data_ptr(), m, n, 0, 1, ps, items[r].data_ptr(), m, 0, 0, mode, 1, 2,
                                         streams[r].cuda_stream)
    torch.cuda.synchronize()
    single = items[0].cpu().numpy().view(ITEM_DTYPE)[0].copy()
    singles_agree = all(bool(x == single) for x in np.concatenate([it.cpu().numpy().view(ITEM_DTYPE) for it in items]))

    for _ in range(calls):      # back to back, no synchronisation in between
        for r in range(world):
            ctxs[r].align_long_cyclic_device(a_ptr[r], dB.data_ptr(), m, n, r, world, ps, items[r].data_ptr(), m, xin[r],
                                             xin[(r + 1) % world], mode, 1, 2, streams[r].cuda_stream)
    torch.cuda.synchronize()
    allitems = np.concatenate([it.cpu().numpy().view(ITEM_DTYPE) for it in items])
    res = multigpu.merge_local_results(allitems) if mode == psa.LOCAL else allitems[multigpu.last_panel_rank(n, world, ps, cols)]
    if mode == psa.LOCAL:
        got, one, want = [(int(x["score"]), int(x["end_i"]), int(x["end_j"])) for x in (res, single)] + [(lin.score, lin.end_i, lin.end_j)]
    else:
        got, one, want = [(int(x["score"]), int(x["t1"]), int(x["t2"]), int(x["t3"])) for x in (res, single)] + [(lin.score, lin.t1, lin.t2, lin.t3)]
    panels = multigpu.panel_owner_ranges(n, world, ps, cols)
    print(json.dumps({"m": m, "n": n, "world": world, "mode": mode, "kc": kc, "panel_strips": ps, "strip_columns": cols,
                      "panels_per_rank": [len(p) for p in panels], "calls": calls, "unaligned_rank": unaligned_rank, "a_offset": a_offset,
                      "got": got, "single_rank": one, "oracle": want, "matches_oracle": got == want,
                      "single_rank_matches_oracle": one == want, "single_runs_agree": singles_agree}), flush=True)
    for r in range(world):
        ctxs[r].xbuf_destroy(xin[r])
        ctxs[r].close()


if __name__ == "__main__":
    main()
