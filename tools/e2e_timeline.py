"""End-to-end A/B of psa_align_batch_packed on the config-2 batch: fills of consecutive chunks serialised or not
(option pack_serial_fills), fixed-stride ops or PSA_OPS_COMPACT; wall time per call (median / min of REPS) and, with
TIMELINE=1, the library's per-chunk GPU timeline (option timing=2, stderr).  PAIRS=1000000 python tools/e2e_timeline.py"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cse305_parallel_sequence_alignment_b200 as psa  # noqa: E402
from cse305_parallel_sequence_alignment_b200 import synth  # noqa: E402

n, L = int(os.environ.get("PAIRS", 1_000_000)), 150
reps = int(os.environ.get("REPS", 12))
A, B = synth.read_pair_batch(n, L, synth.SEED_C2)
pin = lambda x: torch.from_numpy(x).pin_memory().numpy()
a2, b2 = pin(psa.pack_reads_2bit(A).view(np.int32)).view(np.uint32), pin(psa.pack_reads_2bit(B).view(np.int32)).view(np.uint32)
stride = (2 * L + 15) // 16 + 1
items = pin(np.zeros(n * 4, dtype=np.int32)).view(psa.capi.PACKED_ITEM_DTYPE)
ops = pin(np.zeros(n * stride, dtype=np.int32)).view(np.uint32).reshape(n, stride)
ctx = psa.Context(0)
for rnd in range(2):
    for serial, compact in [(s_, c_) for s_ in (0, 1) for c_ in (False, True)]:
        ctx.set_option("pack_serial_fills", serial)
        ts = []
        for rep in range(reps + 2):
            t0 = time.perf_counter()
            ctx.align_batch_packed(a2, b2, L, L, psa.LOCAL, 1, 2, True, items=items, ops=ops, compact=compact)
            if rep >= 2:
                ts.append((time.perf_counter() - t0) * 1e3)
        print(json.dumps({"serial_fills": serial, "compact": compact, "round": rnd, "median_ms": float(np.median(ts)), "min_ms": float(min(ts))}), flush=True)
        if rnd == 1 and os.environ.get("TIMELINE") == "1":
            print(f"---- serial_fills={serial} compact={compact} ----", file=sys.stderr, flush=True)
            ctx.set_option("timing", 2)
            ctx.align_batch_packed(a2, b2, L, L, psa.LOCAL, 1, 2, True, items=items, ops=ops, compact=compact)
            ctx.set_option("timing", 0)
ctx.close()
