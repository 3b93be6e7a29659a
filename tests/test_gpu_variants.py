"""Kernel variants that only an input the other tests never produce selects, each against a plain reference.

A. The systolic kernel (long_systolic = 1) with 1-, 2- and 4-row steps.  The launcher takes 2-row steps whenever A is
   not 4-byte aligned (a sliced tensor, a pair at an odd offset of a batch), and 1-row steps on request; rows are padded
   to the step height, and every ring between strips numbers its rows cumulatively over the calls of a context.
B. sequence_similarity through its three launch shapes (8 lanes per pair up to 512 bytes, 32 lanes up to 8 192, split
   CTAs + a finish kernel above), on hand-placed members at every (A, B) misalignment, around each cut-off of the
   head / aligned words / tail split, and on byte patterns that catch a per-byte count error.
C. Lengths at the long kernels' limit 2^21 - 2, where the 21-bit fields of the local best key come down to 1, and the
   refusal of 2^21 - 1 on every long entry.

Integers must equal the oracle exactly, similarity ratios bit for bit."""
import concurrent.futures
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
from oracle import pyoracle as po
from tests.helpers import mutated_copy, random_dna

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_RANGE = -2
LIMIT = (1 << 21) - 2          # the longest side the long kernels take: i, j <= 2^21 - 2 keep 0x1FFFFF - i >= 1


def new_ctx(**options):
    c = psa.Context(0)
    for k, v in options.items():
        c.set_option(k, v)
    return c


@functools.lru_cache(maxsize=None)
def lin(a, b, mode, g=1, h=2):
    return po.score_linear(a, b, g, h, mode=mode)


def same_score(it, want, mode, tag):
    get = (lambda f: it[f]) if isinstance(it, np.void) else (lambda f: getattr(it, f))
    assert get("score") == want.score, (tag, get("score"), want.score)
    assert (get("end_i"), get("end_j")) == (want.end_i, want.end_j), tag
    if mode == psa.GLOBAL:
        assert (get("t1"), get("t2"), get("t3"), get("end_state")) == (want.t1, want.t2, want.t3, want.end_state), tag


def cuda():
    import torch
    return torch, torch.device("cuda", 0)


def device_bytes(data: bytes, offset=0):
    """A torch uint8 buffer holding `data` at byte `offset` of a fresh allocation; returns (buffer, pointer)."""
    torch, dev = cuda()
    buf = torch.zeros(len(data) + offset + 4, dtype=torch.uint8, device=dev)
    buf[offset:offset + len(data)] = torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).to(dev)
    return buf, buf.data_ptr() + offset


def long_device(ctx, pa, pb, m, n, mode, g=1, h=2):
    """psa_align_long_device score only on a torch side stream -> the record."""
    torch, dev = cuda()
    st = torch.cuda.Stream(device=dev)
    item = torch.zeros(10, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.align_long_device(pa, pb, m, n, item.data_ptr(), 0, 0, mode, g, h, False, st.cuda_stream)
    st.synchronize()
    return item.cpu().numpy().view(ITEM_DTYPE)[0].copy()


# ---- A. systolic row steps ---------------------------------------------------------------------------------------

SMALL_M = [1, 2, 3, 5, 31, 32, 33, 1023, 1025]
STRIP_N = {8: (300, 700), 4: (300, 383)}        # 2 and 3 strips of 32 * KC columns (and > 256: not the short kernel)
WIDE_SHAPES = [(300, 700), (129, 2049), (6000, 9000)]


@functools.lru_cache(maxsize=None)
def systolic_pairs(kc):
    """Random pairs at every shape; then pairs where both sides contain 0x00 (rows past m are read as 0, so a zero
    column byte matches the padding rows)."""
    rng = np.random.default_rng(900 + kc)
    out = []
    for m in SMALL_M:
        for n in STRIP_N[kc]:
            a = random_dna(rng, m)
            out.append((a, mutated_copy(rng, a, n) if (m + n) % 2 else random_dna(rng, n)))
    for m, n in WIDE_SHAPES:
        a = random_dna(rng, m)
        out.append((a, mutated_copy(rng, a, n)))
    zero = np.frombuffer(b"\0ACG", dtype=np.uint8)
    for m, n in [(5, STRIP_N[kc][1]), (33, STRIP_N[kc][0]), (1025, STRIP_N[kc][1])]:
        a = zero[rng.integers(0, 4, size=m)].tobytes()
        b = bytearray(mutated_copy(rng, a, n))
        b[m:] = bytes(n - m) if m < n else b""                 # the columns the padding rows meet: all 0x00
        out.append((a, bytes(b)))
    return out


@pytest.mark.parametrize("kc", [8, 4])
@pytest.mark.parametrize("rb", [4, 2, 1])
def test_systolic_row_steps(rb, kc):
    """RB = 4, 2, 1 (option systolic_rb) and KC = 8, 4, both modes: score, corners, end state and local end cell ==
    the linear-space oracle.  One context per (RB, KC): its rings wrap many laps over the calls."""
    c = new_ctx(long_systolic=1, systolic_kc=kc, systolic_rb=rb)
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            for a, b in systolic_pairs(kc):
                l0 = c.launches
                got = c.align_pair(a, b, mode, traceback=False)
                assert c.launches - l0 == 2, (rb, kc, len(a), len(b))       # one panel + the result kernel
                same_score(got, lin(a, b, mode), mode, (rb, kc, mode, len(a), len(b)))
    finally:
        c.close()


def test_systolic_unaligned_a_through_long_device():
    """psa_align_long_device with A at byte offsets 1, 2, 3 (the launcher falls back to 2-row steps) == the oracle and
    == systolic_rb = 2 on an aligned copy, record for record."""
    rng = np.random.default_rng(31)
    c = new_ctx(long_systolic=1)
    ref = new_ctx(long_systolic=1, systolic_rb=2)
    try:
        for m, n in [(1, 700), (5, 300), (33, 700), (1025, 700), (2001, 555), (6003, 9000)]:
            a = random_dna(rng, m)
            b = mutated_copy(rng, a, n)
            bufb, pb = device_bytes(b)
            bufa0, pa0 = device_bytes(a)
            for mode in (psa.GLOBAL, psa.LOCAL):
                want = long_device(ref, pa0, pb, m, n, mode)
                same_score(want, lin(a, b, mode), mode, (m, n, mode, "rb2 aligned"))
                for off in (1, 2, 3):
                    bufa, pa = device_bytes(a, off)
                    got = long_device(c, pa, pb, m, n, mode)
                    assert got == want, (m, n, mode, off, got, want)
    finally:
        c.close()
        ref.close()


def test_systolic_unaligned_members_of_a_batch():
    """psa_align_batch with <= 8 long score-only pairs of odd lengths: the per-pair loop hands each member to the
    systolic kernel at its own offset of the staged bases, most of them not 4-byte aligned."""
    rng = np.random.default_rng(32)
    lens = [(301, 701), (1023, 333), (5, 515), (777, 1999), (33, 301), (2049, 641), (1, 299)]
    As = [random_dna(rng, m) for m, _ in lens]
    Bs = [mutated_copy(rng, a, n) for a, (_, n) in zip(As, lens)]
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    assert sum(o % 4 != 0 for o in oa) >= 4
    c = new_ctx(long_systolic=1)
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            l0 = c.launches
            items, _ = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=False)
            assert c.launches - l0 == 2 * len(As), mode
            for k, (a, b) in enumerate(zip(As, Bs)):
                same_score(items[k], lin(a, b, mode), mode, (mode, k))
    finally:
        c.close()


def test_systolic_one_context_mixed_step_heights():
    """One context, 14 calls alternating aligned A (4-row steps), A at an odd offset (2-row steps) and systolic_rb = 1,
    m never a multiple of 4: the rings' cumulative row counters are shared by launches of different step heights and
    wrap several 1 024-row laps."""
    rng = np.random.default_rng(33)
    c = new_ctx(long_systolic=1)
    try:
        ms = [1025, 5, 1023, 333, 2050, 517, 1029, 701, 6, 1301, 2, 999, 1031, 13]
        for k, m in enumerate(ms):
            assert m % 4
            n = (300, 700, 555)[k % 3]
            a = random_dna(rng, m)
            b = mutated_copy(rng, a, n) if k % 2 else random_dna(rng, n)
            kind = k % 3
            c.set_option("systolic_rb", 1 if kind == 2 else 4)
            bufa, pa = device_bytes(a, 1 + k % 3 if kind == 1 else 0)
            bufb, pb = device_bytes(b)
            for mode in (psa.GLOBAL, psa.LOCAL):
                same_score(long_device(c, pa, pb, m, n, mode), lin(a, b, mode), mode, (k, m, n, kind, mode))
    finally:
        c.close()


@pytest.mark.parametrize("rb", [4, 1])
def test_systolic_short_a_across_panels(rb):
    """m = 1 ... 5 on fresh contexts, one-strip panels (the cyclic entry with one rank): consecutive panels hand over
    through the context's own boundary buffers, whose capacity follows m."""
    rng = np.random.default_rng(34)
    for m in (1, 2, 3, 5):
        for mode in (psa.GLOBAL, psa.LOCAL):
            c = new_ctx(systolic_rb=rb)
            try:
                a = random_dna(rng, m)
                b = random_dna(rng, 700)
                bufa, pa = device_bytes(a)
                bufb, pb = device_bytes(b)
                torch, dev = cuda()
                item = torch.zeros(10, dtype=torch.int32, device=dev)
                torch.cuda.synchronize()
                l0 = c.launches
                c.align_long_cyclic_device(pa, pb, m, 700, 0, 1, 1, item.data_ptr(), m, 0, 0, mode)
                torch.cuda.synchronize()
                assert c.launches - l0 == 3 + 1, (m, mode)        # three 256-column panels + the result kernel
                same_score(item.cpu().numpy().view(ITEM_DTYPE)[0], lin(a, b, mode), mode, (rb, m, mode))
            finally:
                c.close()


def test_cyclic_ranks_one_unaligned():
    """The cyclic entry with 2 and 3 ranks sharing one device (tools/cyclic_one_gpu.py), one rank's A at an odd offset:
    its panels take 2-row steps and hand rows to ranks that take 4-row steps.  m = 9 001 (not a multiple of 4).  The
    merged result == the single-rank run == the oracle.  In a child process with a time limit, so that a ring protocol
    error fails instead of hanging the run."""
    variants = [{"world": 2, "panel_strips": 8, "kc": 8, "mode": 1, "unaligned_rank": 1, "a_offset": 1},
                {"world": 3, "panel_strips": 8, "kc": 8, "mode": 0, "unaligned_rank": 0, "a_offset": 2},
                {"world": 3, "panel_strips": 5, "kc": 4, "mode": 1, "unaligned_rank": 2, "a_offset": 3}]
    env = dict(os.environ, M="9001", N="20000", CALLS="3", VARIANTS=json.dumps(variants))
    run = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cyclic_one_gpu.py")], env=env, capture_output=True,
                         text=True, timeout=240)
    assert run.returncode == 0, run.stderr[-2000:]
    outs = [json.loads(x) for x in run.stdout.splitlines() if x.startswith("{")]
    assert len(outs) == len(variants)
    for out in outs:
        assert out["matches_oracle"] and out["single_rank_matches_oracle"] and out["single_runs_agree"], out
        assert min(out["panels_per_rank"]) >= 2, out


# ---- B. similarity -------------------------------------------------------------------------------------------------

KINDS = ["zero", "ff", "eq", "diff", "every4", "rand", "zero_ff"]


def sim_bytes(rng, kind, la, lb, k):
    """Two members whose first min(la, lb) bytes follow `kind`; the rest is random."""
    L = min(la, lb)
    tail_a, tail_b = rng.integers(0, 256, size=la - L, dtype=np.uint8), rng.integers(0, 256, size=lb - L, dtype=np.uint8)
    if kind == "zero":
        x = y = np.zeros(L, np.uint8)
    elif kind == "ff":
        x = y = np.full(L, 0xFF, np.uint8)
    elif kind == "zero_ff":
        x, y = np.zeros(L, np.uint8), np.full(L, 0xFF, np.uint8)
    elif kind == "eq":
        x = y = rng.integers(0, 256, size=L, dtype=np.uint8)
    elif kind == "diff":
        x = rng.integers(0, 256, size=L, dtype=np.uint8)
        y = x ^ np.uint8(1 + k % 255)
    elif kind == "every4":                                  # equal except every 4th byte (phase varies)
        x = rng.integers(0, 256, size=L, dtype=np.uint8)
        y = x.copy()
        y[k % 4::4] ^= np.uint8(0x40)
    else:
        x = rng.integers(0, 4, size=L, dtype=np.uint8)
        y = np.where(rng.random(L) < 0.5, x, rng.integers(0, 4, size=L, dtype=np.uint8)).astype(np.uint8)
    return np.concatenate([x, tail_a]), np.concatenate([y, tail_b])


class Layout:
    """One base array built by hand: members at chosen offsets mod 4, random filler (gaps) between them."""

    def __init__(self, rng):
        self.rng, self.parts, self.size = rng, [], 0

    def put(self, data, mod):
        gap = int(self.rng.integers(0, 6))
        gap += (mod - (self.size + gap)) % 4
        self.parts.append(self.rng.integers(0, 256, size=gap, dtype=np.uint8))
        off = self.size + gap
        self.parts.append(np.asarray(data, dtype=np.uint8))
        self.size = off + len(data)
        return off

    def bytes(self):
        self.parts.append(self.rng.integers(0, 256, size=5, dtype=np.uint8))
        return np.concatenate(self.parts) if self.parts else np.zeros(1, np.uint8)


class SimBatch:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.A, self.B = Layout(self.rng), Layout(self.rng)
        self.oa, self.la, self.ob, self.lb = [], [], [], []
        self.k = 0

    def add(self, la, lb, ma, mb, kind=None):
        x, y = sim_bytes(self.rng, kind or KINDS[self.k % len(KINDS)], la, lb, self.k)
        self.k += 1
        self.oa.append(self.A.put(x, ma)); self.la.append(la)
        self.ob.append(self.B.put(y, mb)); self.lb.append(lb)

    def every_alignment(self, lengths):
        """L = min(len_a, len_b) over `lengths` at all 16 (off_a mod 4, off_b mod 4); the longer side varies."""
        for L in lengths:
            for ma in range(4):
                for mb in range(4):
                    extra = (self.k * 7) % 5
                    self.add(L + (extra if self.k % 2 else 0), L + (0 if self.k % 2 else extra), ma, mb)

    def around_cutoffs(self, cut, width=12):
        """Lengths head + cut - 4 ... head + cut + width for every head = (4 - off_a mod 4) mod 4."""
        for ma in range(4):
            head = (4 - ma) % 4
            for mb in range(4):
                for L in range(max(0, head + cut - 4), head + cut + width, 3):
                    self.add(L, L + (mb & 1), ma, mb)

    def finish(self, extra_pairs=True):
        a, b = self.A.bytes(), self.B.bytes()
        oa, la, ob, lb = (np.array(v, dtype=t) for v, t in ((self.oa, np.int64), (self.la, np.int32), (self.ob, np.int64), (self.lb, np.int32)))
        if extra_pairs and len(oa) > 8:
            # members that overlap another member, and two pairs that share one sequence
            oa = np.concatenate([oa, [oa[3] + 2, oa[5], oa[7]]])
            la = np.concatenate([la, [max(0, int(la[3]) - 2), la[5], la[7]]]).astype(np.int32)
            ob = np.concatenate([ob, [ob[4] + 1, ob[5], ob[7] + 1]])
            lb = np.concatenate([lb, [max(0, int(lb[4]) - 1), lb[5], max(0, int(lb[7]) - 1)]]).astype(np.int32)
        return a, oa, la, b, ob, lb


def sim_expected(a, oa, la, b, ob, lb):
    out = np.zeros(len(la), dtype=np.float64)
    for k in range(len(la)):
        L = int(min(la[k], lb[k]))
        eq = int(np.count_nonzero(a[oa[k]:oa[k] + L] == b[ob[k]:ob[k] + L]))
        mx = int(max(la[k], lb[k]))
        out[k] = eq / mx if mx else 0.0
    return out


def sim_check(ctx, batch, launches, tag):
    a, oa, la, b, ob, lb = batch
    l0 = ctx.launches
    got = ctx.similarity_batch(a, oa, la, b, ob, lb)
    assert ctx.launches - l0 == launches, tag
    want = sim_expected(*batch)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, (tag, [(int(k), int(oa[k]) % 4, int(ob[k]) % 4, int(la[k]), int(lb[k]), got[k], want[k]) for k in bad[:6]])
    return got


def small_batch(seed, top, cutoffs):
    """L = 0 ... 40 at every alignment, the cut-offs given, and one pair whose longer member is exactly `top`."""
    sb = SimBatch(seed)
    sb.every_alignment(range(0, 41))
    for cut in cutoffs:
        sb.around_cutoffs(cut)
    sb.add(top, top - 3, 1, 2)
    sb.add(top - 7, top, 3, 0, "every4")
    batch = sb.finish()
    assert max(int(batch[2].max()), int(batch[5].max())) == top
    return batch


@pytest.fixture(scope="module")
def sim_ctx():
    c = psa.Context(0)
    yield c
    c.close()


# head + 8: the first length with aligned words; 4 + 4 words * lanes * 4 B: one full round of four words in flight
# (8 lanes: 128 B, 32 lanes: 512 B, a 256-thread split CTA: 4 096 B)
@pytest.mark.parametrize("top,cutoffs", [(512, (8, 4 + 128, 4 + 256)), (513, (8, 4 + 128)),
                                                  (8192, (8, 4 + 512, 4 + 1024)), (8193, (8, 4 + 512, 4 + 4096))],
                         ids=["8_lanes_512", "32_lanes_513", "32_lanes_8192", "split_8193"])
def test_similarity_launch_shapes(sim_ctx, top, cutoffs):
    """The batch's largest length picks the kernel: <= 512 the 8-lane kernel, <= 8 192 the 32-lane kernel, above that
    the split kernel + finish kernel (two launches)."""
    sim_check(sim_ctx, small_batch(top, top, cutoffs), 1 if top <= 8192 else 2, top)


def test_similarity_split_slices(sim_ctx):
    """Split-kernel slice counts from 1 to many: one 4 MB pair, 3 pairs, a batch whose 40 000-byte member makes three
    16 384-byte slices per pair with lengths around the slice size, and enough pairs that 2 * cap / n_pairs is 1."""
    rng = np.random.default_rng(40)
    sb = SimBatch(41)
    sb.add(4 << 20, (4 << 20) - 5, 1, 3, "rand")
    sim_check(sim_ctx, sb.finish(), 2, "one 4 MB pair")
    sb = SimBatch(42)
    sb.add(4 << 20, 1 << 20, 0, 1, "every4")
    sb.add((1 << 20) + 3, (1 << 20) + 3, 2, 3, "rand")
    sb.add(17000, 16999, 3, 2, "eq")
    sim_check(sim_ctx, sb.finish(), 2, "3 pairs")
    sb = SimBatch(43)
    sb.every_alignment(range(0, 41, 5))
    for L in (16380, 16383, 16384, 16385, 16388, 16392, 32769):
        for ma, mb in ((0, 0), (1, 2), (3, 1), (2, 3)):
            sb.add(L, L + ma, ma, mb)
    sb.around_cutoffs(4 + 4096, width=6)
    sb.add(40000, 39999, 1, 1, "rand")
    sim_check(sim_ctx, sb.finish(), 2, "three slices")
    sb = SimBatch(44)
    for k in range(2400):
        L = int(rng.integers(16000, 20000))
        sb.add(L, L - k % 3, k % 4, (k // 4) % 4)
    sim_check(sim_ctx, sb.finish(), 2, "2 400 pairs")


def fixed_150(n_pairs, seed):
    rng = np.random.default_rng(seed)
    A = rng.integers(0, 4, size=(n_pairs, 150), dtype=np.uint8)
    B = np.where(rng.random((n_pairs, 150)) < 0.7, A, rng.integers(0, 4, size=(n_pairs, 150), dtype=np.uint8)).astype(np.uint8)
    off = np.arange(n_pairs, dtype=np.int64) * 150
    ln = np.full(n_pairs, 150, dtype=np.int32)
    want = np.count_nonzero(A == B, axis=1) / 150
    return A.reshape(-1), off, ln, B.reshape(-1), off.copy(), ln.copy(), want


def test_similarity_grid_stride_and_device_entry(sim_ctx):
    """100 000 x 150 bp: more than 8 * SMs * 32 pairs, so the 8-lane kernel's CTAs loop.  The device entry on a torch
    side stream == the host entry; an inflated max_len (513, 9 000) runs the 32-lane and the split kernel on the same
    data with identical results."""
    torch, dev = cuda()
    a, oa, la, b, ob, lb, want = fixed_150(100_000, 50)
    l0 = sim_ctx.launches
    host = sim_ctx.similarity_batch(a, oa, la, b, ob, lb)
    assert sim_ctx.launches - l0 == 1
    assert np.array_equal(host, np.array([float(x) for x in want])), np.flatnonzero(host != want)[:8]
    st = torch.cuda.Stream(device=dev)
    t = [torch.from_numpy(x).to(dev) for x in (a, oa, la, b, ob, lb)]
    torch.cuda.synchronize()
    for max_len, launches in ((150, 1), (513, 1), (9000, 2)):
        out = torch.full((len(la),), -1.0, dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        l0 = sim_ctx.launches
        sim_ctx.similarity_batch_device(*(x.data_ptr() for x in t), len(la), max_len, out.data_ptr(), st.cuda_stream)
        assert sim_ctx.launches - l0 == launches, max_len
        st.synchronize()
        assert np.array_equal(out.cpu().numpy(), host), max_len


def test_similarity_device_entry_hand_layout(sim_ctx):
    """The hand-placed 512-byte batch through the device entry at max_len 512, 513 and 9 000: one result."""
    torch, dev = cuda()
    batch = small_batch(77, 512, (8, 4 + 128))
    host = sim_check(sim_ctx, batch, 1, "host")
    st = torch.cuda.Stream(device=dev)
    t = [torch.from_numpy(x).to(dev) for x in batch]
    for max_len, launches in ((512, 1), (513, 1), (9000, 2)):
        out = torch.full((len(batch[2]),), -1.0, dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        l0 = sim_ctx.launches
        sim_ctx.similarity_batch_device(*(x.data_ptr() for x in t), len(batch[2]), max_len, out.data_ptr(), st.cuda_stream)
        assert sim_ctx.launches - l0 == launches, max_len
        st.synchronize()
        assert np.array_equal(out.cpu().numpy(), host), max_len


# ---- C. lengths at the limit ---------------------------------------------------------------------------------------

LIMIT_SHAPES = [(LIMIT, 257), (LIMIT, 300), (257, LIMIT), (300, LIMIT)]


@functools.lru_cache(maxsize=None)
def limit_pair(m, n, mode):
    """Local: the short side is an exact copy of the long side's last bases, so the best cell is unique and sits at
    i or j = 2^21 - 2.  Global: the short side is a mutated copy of a stretch in the middle of the long side."""
    rng = np.random.default_rng(m * 3 + n + mode)
    long_, short = max(m, n), min(m, n)
    x = random_dna(rng, long_)
    if mode == psa.LOCAL:
        y = x[-short:]
    else:
        mid = long_ // 2 + 7
        y = mutated_copy(rng, x[mid:mid + short], short)
    return (x, y) if m > n else (y, x)


@pytest.fixture(scope="module")
def limit_oracle():
    """score_linear of every limit pair (seconds each), computed once, in parallel threads."""
    keys = [(m, n, mode) for m, n in LIMIT_SHAPES for mode in (psa.GLOBAL, psa.LOCAL)]
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(keys)) as ex:
        futs = {k: ex.submit(po.score_linear, *limit_pair(*k), 1, 2, k[2]) for k in keys}
        return {k: f.result() for k, f in futs.items()}


def local_expect(m, n, want):
    """The copied stretch: end cell (m, n), score = the short length, a run of diagonal columns."""
    short = min(m, n)
    assert (want.score, want.end_i, want.end_j) == (short, m, n)
    return short


def rescore(a, b, ops, start_i, start_j, g=1, h=2):
    """Score of the global path: the border run the traceback leaves out, then `ops` (1 diagonal, 2 gap in A,
    3 gap in B).  Every base of both sides must be consumed exactly once."""
    assert start_i == 1 or start_j == 1
    full = np.concatenate([np.full(start_i - 1, 3, np.uint8), np.full(start_j - 1, 2, np.uint8), np.frombuffer(ops, np.uint8)])
    i = np.cumsum(full != 2)
    j = np.cumsum(full != 3)
    assert i[-1] == len(a) and j[-1] == len(b)
    diag = full == 1
    av, bv = np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8)
    matches = int(np.count_nonzero(av[i[diag] - 1] == bv[j[diag] - 1]))
    gaps = ~diag
    opens = gaps & (full != np.concatenate([[0], full[:-1]]))
    return matches - g * int(np.count_nonzero(gaps)) - h * int(np.count_nonzero(opens))


@pytest.mark.parametrize("shape", LIMIT_SHAPES, ids=[f"{m}x{n}" for m, n in LIMIT_SHAPES])
def test_limit_score_only_routes(limit_oracle, shape):
    """align_pair score only on the default geometry, geometries 0, 2, 6, 7 and the systolic kernel; the int32 long
    batch (pack = 0, nine members so that the batch kernel runs)."""
    m, n = shape
    routes = [("default", {}), ("geo0", {"long_geometry": 0}), ("geo2", {"long_geometry": 2}), ("geo6", {"long_geometry": 6}),
              ("geo7", {"long_geometry": 7}), ("systolic", {"long_systolic": 1})]
    for name, opts in routes:
        c = new_ctx(**opts)
        try:
            for mode in (psa.GLOBAL, psa.LOCAL):
                a, b = limit_pair(m, n, mode)
                want = limit_oracle[(m, n, mode)]
                if mode == psa.LOCAL:
                    local_expect(m, n, want)
                same_score(c.align_pair(a, b, mode, traceback=False), want, mode, (shape, name, mode))
        finally:
            c.close()
    rng = np.random.default_rng(m + 2 * n)
    c = new_ctx(pack=0)
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            a, b = limit_pair(m, n, mode)
            As, Bs = [a], [b]
            for _ in range(8):                       # small members keep the short side's bound
                x = random_dna(rng, int(rng.integers(200, min(m, 300) + 1) if m < n else rng.integers(300, 2000)))
                y = mutated_copy(rng, x, int(rng.integers(300, 2000)) if m < n else int(rng.integers(200, min(n, 300) + 1)))
                As.append(x); Bs.append(y)
            ba, oa, la = psa.pack_pairs(As)
            bb, ob, lb = psa.pack_pairs(Bs)
            l0 = c.launches
            items, _ = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=False)
            assert c.launches - l0 == 1, (shape, mode)
            same_score(items[0], limit_oracle[(m, n, mode)], mode, (shape, "batch", mode))
            for k in range(1, len(As)):
                same_score(items[k], lin(As[k], Bs[k], mode), mode, (shape, "batch", mode, k))
    finally:
        c.close()


def device_batch_tb(ctx, As, Bs, mode):
    """psa_align_batch_device with traceback, on a torch side stream."""
    torch, dev = cuda()
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    n = len(As)
    stride = (int(la.max()) + int(lb.max()) + 15) // 16 + 1
    st = torch.cuda.Stream(device=dev)
    t = [torch.from_numpy(x).to(dev) for x in (ba, oa, la, bb, ob, lb)]
    items = torch.zeros(n * 10, dtype=torch.int32, device=dev)
    ops = torch.zeros(n * stride, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.align_batch_device(*(x.data_ptr() for x in t), n, int(la.max()), int(lb.max()), items.data_ptr(), ops.data_ptr(),
                           stride, mode, 1, 2, True, st.cuda_stream)
    st.synchronize()
    return items.cpu().numpy().view(ITEM_DTYPE).copy(), ops.cpu().numpy().view(np.uint32).reshape(n, stride).copy()


@pytest.mark.parametrize("shape", [(LIMIT, 300), (300, LIMIT)], ids=["long_a", "long_b"])
def test_limit_traceback_routes(limit_oracle, shape):
    """align_pair with traceback, band recompute on and off, and a 16-member device traceback batch with the limit pair
    as member 0.  Local: the copied stretch (diagonal columns ending at 2^21 - 2) exactly.  Global: the full tables do
    not fit, so the ops must re-score to the oracle's corner value, and all three routes must give the same ops."""
    m, n = shape
    rng = np.random.default_rng(m + 3 * n)
    for mode in (psa.GLOBAL, psa.LOCAL):
        a, b = limit_pair(m, n, mode)
        want = limit_oracle[(m, n, mode)]
        results = []
        for band in (1, 0):
            c = new_ctx(long_band=band)
            try:
                got = c.align_pair(a, b, mode)
            finally:
                c.close()
            same_score(got, want, mode, (shape, mode, band))
            results.append((got.start_i, got.start_j, got.ops))
            if mode == psa.GLOBAL:
                assert rescore(a, b, got.ops, got.start_i, got.start_j) == want.score, (shape, band)
                assert got.row_a.replace(b"-", b"")[-50:] == a[-50:] and got.row_b.replace(b"-", b"")[-50:] == b[-50:]
        As, Bs = [a], [b]
        for _ in range(15):
            x = random_dna(rng, int(rng.integers(200, 301)) if m < n else int(rng.integers(300, 1500)))
            As.append(x)
            Bs.append(mutated_copy(rng, x, int(rng.integers(300, 1500)) if m < n else int(rng.integers(200, 301))))
        c = psa.Context(0)
        try:
            items, ops = device_batch_tb(c, As, Bs, mode)
        finally:
            c.close()
        it = items[0]
        same_score(it, want, mode, (shape, mode, "batch"))
        results.append((int(it["start_i"]), int(it["start_j"]), psa.unpack_ops(ops[0], int(it["aln_len"]))))
        assert results[0] == results[1] == results[2], (shape, mode, [r[:2] + (len(r[2]),) for r in results])
        if mode == psa.LOCAL:
            short = local_expect(m, n, want)
            assert results[0] == ((m - short + 1, 1, b"\x01" * short) if m > n else (1, n - short + 1, b"\x01" * short))
        for k in range(1, 16):
            w = po.align(As[k], Bs[k], 1, 2, mode=mode)
            same_score(items[k], w, mode, (shape, mode, k))
            assert psa.unpack_ops(ops[k], int(items[k]["aln_len"])) == w.ops, (shape, mode, k)


@pytest.mark.parametrize("shape", [(LIMIT, 300), (257, LIMIT)], ids=["long_a", "long_b"])
def test_limit_partitioned(limit_oracle, shape):
    """psa_align_long_partitioned with 5 pieces: a complete alignment that re-scores to the oracle's optimum."""
    m, n = shape
    a, b = limit_pair(m, n, psa.GLOBAL)
    c = psa.Context(0)
    try:
        got, crossings = c.align_long_partitioned(a, b, 5, 1, 2)
    finally:
        c.close()
    want = limit_oracle[(m, n, psa.GLOBAL)]
    assert got.score == want.score
    assert got.row_a.replace(b"-", b"") == a and got.row_b.replace(b"-", b"") == b
    av, bv = np.frombuffer(got.row_a, np.uint8), np.frombuffer(got.row_b, np.uint8)
    ops = np.where(av == 0x2D, 2, np.where(bv == 0x2D, 3, 1)).astype(np.uint8).tobytes()
    assert rescore(a, b, ops, 1, 1) == want.score
    assert 1 <= len(crossings) <= 4 and crossings == sorted(crossings)


def test_limit_refusals():
    """2^21 - 1 is refused with PSA_ERR_RANGE by align_pair (long path), psa_align_long_device,
    psa_align_long_partitioned and psa_align_long_cyclic_device; after each refusal the context still answers right."""
    torch, dev = cuda()
    rng = np.random.default_rng(21)
    over = LIMIT + 1
    big = random_dna(rng, over)
    a = random_dna(rng, 700)
    b = mutated_copy(rng, a, 900)
    bufbig, pbig = device_bytes(big)
    bufa, pa = device_bytes(a)
    bufb, pb = device_bytes(b)
    item = torch.zeros(10, dtype=torch.int32, device=dev)
    small = random_dna(rng, 300)
    bufs, ps = device_bytes(small)
    c = psa.Context(0)
    try:
        def still_right(tag):
            for mode in (psa.GLOBAL, psa.LOCAL):
                same_score(c.align_pair(a, b, mode, traceback=False), lin(a, b, mode), mode, (tag, mode))
            same_score(long_device(c, pa, pb, 700, 900, psa.LOCAL), lin(a, b, psa.LOCAL), psa.LOCAL, (tag, "device"))

        calls = [("pair", lambda: c.align_pair(big, small, psa.GLOBAL, traceback=False)),
                 ("pair_t", lambda: c.align_pair(small, big, psa.LOCAL, traceback=False)),
                 ("pair_tb", lambda: c.align_pair(big, small, psa.GLOBAL)),
                 ("device", lambda: c.align_long_device(pbig, ps, over, 300, item.data_ptr(), 0, 0, psa.LOCAL)),
                 ("device_t", lambda: c.align_long_device(ps, pbig, 300, over, item.data_ptr(), 0, 0, psa.GLOBAL)),
                 ("partitioned", lambda: c.align_long_partitioned(big, small, 5)),
                 ("partitioned_t", lambda: c.align_long_partitioned(small, big, 5)),
                 ("cyclic", lambda: c.align_long_cyclic_device(pbig, ps, over, 300, 0, 1, 8, item.data_ptr(), over)),
                 ("cyclic_t", lambda: c.align_long_cyclic_device(ps, pbig, 300, over, 0, 1, 8, item.data_ptr(), 300))]
        for name, call in calls:
            with pytest.raises(psa.PsaError) as e:
                call()
                torch.cuda.synchronize()
            assert e.value.code == ERR_RANGE, name
            still_right(name)
    finally:
        c.close()
