"""GPU parity of the long-pair path (row-block wavefront, checkpointed traceback, long batches)
through the C-ABI against the oracle and the reference's golden vectors."""
import hashlib
import json
import os
import random

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200 import synth
from oracle import pyoracle as po
from tests.helpers import GOLDEN, dataset, mutated_copy, random_dna

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = psa.Context(0)
    yield c
    c.close()


def _same(got, want, local=False):
    assert got.score == want.score
    if not local:
        assert (got.t1, got.t2, got.t3, got.end_state) == (want.t1, want.t2, want.t3, want.end_state)
    assert (got.end_i, got.end_j) == (want.end_i, want.end_j)
    assert got.ops == want.ops
    assert (got.start_i, got.start_j) == (want.start_i, want.start_j)
    assert (got.row_a, got.row_b) == (want.row_a, want.row_b)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_tile_boundaries_vs_oracle(ctx, mode):
    """Sizes around the 128-row / 256-column tile edges, with traceback."""
    rng = np.random.default_rng(5 + mode)
    rnd = random.Random(5 + mode)
    for (m, n) in [(1, 257), (127, 257), (128, 256 + 1), (129, 300), (255, 511), (256, 512), (257, 513), (300, 300),
                   (640, 700), (1000, 1030), (383, 1025)]:
        a = random_dna(rng, m)
        b = mutated_copy(rng, a, n) if rnd.random() < 0.7 else random_dna(rng, n)
        g, h = rnd.choice([(1, 2), (1, 2), (2, 1), (1, 0)])
        _same(ctx.align_pair(a, b, mode, g, h), po.align(a, b, g, h, mode=mode), local=(mode == psa.LOCAL))


def test_m_greater_than_n_long(ctx):
    rng = np.random.default_rng(9)
    a = random_dna(rng, 900)
    b = mutated_copy(rng, a[100:500], 400)
    for mode in (psa.GLOBAL, psa.LOCAL):
        _same(ctx.align_pair(a, b, mode, 1, 2), po.align(a, b, 1, 2, mode=mode), local=(mode == psa.LOCAL))


def test_dataset_kats(ctx):
    """SURVEY 8c G6: dataset prefixes up to 13 327 bp, rows checked by md5 against the reference."""
    names, seqs = dataset()
    for case in json.load(open(os.path.join(GOLDEN, "kat.json"))):
        if case.get("L", 0) <= 256:
            continue
        a, b = seqs[case["rec_a"]][:case["L"]].encode(), seqs[case["rec_b"]][:case["L"]].encode()
        got = ctx.align_pair(a, b, psa.GLOBAL, case["g"], case["h"])
        assert [got.t1, got.t2, got.t3] == case["corner"] and got.end_state == case["end_state"], case["name"]
        assert len(got.ops) == case["cols"]
        assert (got.ops.count(1), got.ops.count(2), got.ops.count(3)) == (case["n_t1"], case["n_t2"], case["n_t3"])
        assert hashlib.md5(got.row_a + b"\n" + got.row_b + b"\n").hexdigest() == case["md5"], case["name"]


def test_config3_10k_mutated_copy(ctx):
    """BASELINE config 3: 10 kbp x 10 kbp mutated copy, full alignment, checkpointed traceback."""
    A, B = synth.mutated_pair(10000, synth.SEED_C3)
    a, b = A.tobytes(), B.tobytes()
    got = ctx.align_pair(a, b, psa.GLOBAL, 1, 2)
    want = po.align(a, b, 1, 2)
    _same(got, want)
    gotl = ctx.align_pair(a, b, psa.LOCAL, 1, 2)
    wantl = po.align(a, b, 1, 2, mode=po.LOCAL)
    _same(gotl, wantl, local=True)


def test_single_long_score_only(ctx):
    rng = np.random.default_rng(21)
    a = random_dna(rng, 5000)
    b = mutated_copy(rng, a, 7000)
    for mode in (psa.GLOBAL, psa.LOCAL):
        got = ctx.align_pair(a, b, mode, 1, 2, traceback=False)
        lin = po.score_linear(a, b, 1, 2, mode=mode)
        assert got.score == lin.score and (got.end_i, got.end_j) == (lin.end_i, lin.end_j)
        if mode == psa.GLOBAL:
            assert (got.t1, got.t2, got.t3, got.end_state) == (lin.t1, lin.t2, lin.t3, lin.end_state)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_long_batch_score_only(ctx, mode):
    """Config 5 shape at reduced size: many long pairs, score + end cell, one warp per pair."""
    rng = np.random.default_rng(33 + mode)
    As, Bs = [], []
    for k in range(40):
        m = int(rng.integers(300, 1600))
        n = int(rng.integers(m, m + 300))
        a = random_dna(rng, m)
        As.append(a)
        Bs.append(mutated_copy(rng, a, n) if k % 3 else random_dna(rng, n))
    As.append(b""); Bs.append(random_dna(rng, 400))       # ragged / empty members
    As.append(random_dna(rng, 400)); Bs.append(b"")
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    items, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=False)
    for k in range(len(As)):
        lin = po.score_linear(As[k], Bs[k], 1, 2, mode=mode)
        it = items[k]
        assert it["score"] == lin.score, k
        assert (it["end_i"], it["end_j"]) == (lin.end_i, lin.end_j), k
        if mode == psa.GLOBAL:
            assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (lin.t1, lin.t2, lin.t3, lin.end_state), k


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_config5_shape_packed_long(ctx, mode):
    """Config 5 at full pair size (5 kbp x 5 kbp, a few pairs): packed .S16x2 strip kernel, with a
    non-ACGT member and ragged lengths mixed in (int32 fallback), against the linear oracle."""
    A, B = synth.read_pair_batch(6, 5000, synth.SEED_C5)
    As = [A[k].tobytes() for k in range(6)]
    Bs = [B[k].tobytes() for k in range(6)]
    rng = np.random.default_rng(77)
    As.append(random_dna(rng, 4500)); Bs.append(mutated_copy(rng, As[-1], 4800))
    As.append(As[0].replace(b"A", b"N")); Bs.append(Bs[0])            # not plain ACGT
    As.append(random_dna(rng, 700)); Bs.append(random_dna(rng, 5000))
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    items, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=False)
    for k in range(len(As)):
        lin = po.score_linear(As[k], Bs[k], 1, 2, mode=mode)
        it = items[k]
        assert it["score"] == lin.score and (it["end_i"], it["end_j"]) == (lin.end_i, lin.end_j), k
        if mode == psa.GLOBAL:
            assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (lin.t1, lin.t2, lin.t3, lin.end_state), k


@pytest.fixture(params=[8, 4])
def systolic_ctx(request):
    c = psa.Context(0)
    c.set_option("long_systolic", 1)
    c.set_option("systolic_kc", request.param)          # columns per lane: 8 is the default, 4 the narrow variant
    assert c.long_strip_columns == 32 * request.param
    yield c
    c.close()


def test_systolic_kernel_matches_oracle(systolic_ctx):
    """The column-stationary systolic kernel forced onto small pairs (option long_systolic=1): rings between
    strips, checkpoints for the traceback -- same answers as the oracle."""
    ctx = systolic_ctx
    rng = np.random.default_rng(123)
    for (m, n) in [(300, 700), (1000, 1030), (129, 2049), (2500, 2400)]:
        a = random_dna(rng, m)
        b = mutated_copy(rng, a, n)
        for mode in (psa.GLOBAL, psa.LOCAL):
            _same(ctx.align_pair(a, b, mode, 1, 2), po.align(a, b, 1, 2, mode=mode), local=(mode == psa.LOCAL))
    a = random_dna(rng, 6000)
    b = mutated_copy(rng, a, 9000)
    for mode in (psa.GLOBAL, psa.LOCAL):
        got = ctx.align_pair(a, b, mode, 1, 2, traceback=False)
        lin = po.score_linear(a, b, 1, 2, mode=mode)
        assert got.score == lin.score and (got.end_i, got.end_j) == (lin.end_i, lin.end_j)


@pytest.mark.parametrize("n,period", [(700, 256), (1500, 512), (1500, 256)])
def test_packed_long_tie_break_across_strips(ctx, n, period):
    """Local end cell = smallest i, then smallest j.  Backgrounds that never match (A is all 'A', B all 'C')
    carry two different 48-base motifs over {G,T}: both diagonals reach T1 = 48, and since a mismatch
    costs 0 they stay there.  The motif at the smaller rows sits `period` columns further right, i.e. in
    a later column strip but in the columns of the same lane (strips are 256 or 512 columns wide) -- a
    per-lane best that only remembers the first maximum it meets reports the wrong cell."""
    rng = np.random.default_rng(n + period)
    gt = np.frombuffer(b"GT", dtype=np.uint8)
    As, Bs = [], []
    for k in range(70):
        m1 = gt[rng.integers(0, 2, size=48)].tobytes()
        m2 = gt[rng.integers(0, 2, size=48)].tobytes()
        a = bytearray(b"A" * 640)
        b = bytearray(b"C" * n)
        c1 = int(rng.integers(10, 150))                 # motif 1: large row, early column
        r_big, r_small = 400 + int(rng.integers(0, 100)), 60 + int(rng.integers(0, 100))
        a[r_big:r_big + 48] = m1
        b[c1:c1 + 48] = m1
        a[r_small:r_small + 48] = m2                    # motif 2: small row, `period` columns later
        b[c1 + period:c1 + period + 48] = m2
        As.append(bytes(a)); Bs.append(bytes(b))
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    items, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.LOCAL, 1, 2, traceback=False)
    ties = 0
    for k in range(len(As)):
        lin = po.score_linear(As[k], Bs[k], 1, 2, mode=psa.LOCAL)
        it = items[k]
        assert it["score"] == lin.score, k
        assert (it["end_i"], it["end_j"]) == (lin.end_i, lin.end_j), (k, lin.score)
        ties += lin.score == 48
    assert ties > 30          # the construction really produces the two-way tie most of the time


def test_typed_subproblems_long(ctx):
    """Start/end types (SURVEY 8 f-2) on the long-pair kernels: every (start, end) combination on pairs
    that span several row blocks and column strips, checkpointed traceback, against the oracle."""
    rng = np.random.default_rng(99)
    for st in (-1, -2, -3, 1, 2, 3):
        for et in (-1, -2, -3, 1, 2, 3):
            m = int(rng.integers(140, 700))
            n = int(rng.integers(260, 900))
            a = random_dna(rng, m)
            b = mutated_copy(rng, a, n, sub=0.1, ins=0.03, dele=0.03) if (st + et) % 2 else random_dna(rng, n)
            g, h = [(1, 2), (2, 1), (1, 0), (0, 3)][int(rng.integers(0, 4))]
            want = po.align(a, b, g, h, start_type=st, end_type=et)
            got = ctx.align_pair(a, b, psa.GLOBAL, g, h, start_type=st, end_type=et)
            assert (got.t1, got.t2, got.t3, got.end_state) == (want.t1, want.t2, want.t3, want.end_state), (st, et, m, n)
            assert got.ops == want.ops and (got.row_a, got.row_b) == (want.row_a, want.row_b), (st, et, m, n)
            assert (got.start_i, got.start_j) == (want.start_i, want.start_j)
    # a partition with one piece wider than 256 columns: pieces run one after the other
    a = random_dna(rng, 1500)
    b = mutated_copy(rng, a, 1500, sub=0.05)
    whole = po.align(a, b, 1, 2)
    i, j, nodes = whole.start_i, whole.start_j, []
    for k, t in enumerate(whole.ops):
        if k:
            i += t != 2; j += t != 3
        nodes.append((i, j, t))
    points = [(0, 0, -1), nodes[100], nodes[900], nodes[1100], (1500, 1500, 1)]
    ops = ra = rb = b""
    for (i0, j0, t0), (i1, j1, t1) in zip(points[:-1], points[1:]):
        piece = po.align(a[i0:i1], b[j0:j1], 1, 2, start_type=t0, end_type=-t1)
        ops += piece.ops; ra += piece.row_a; rb += piece.row_b
    got = ctx.align_partition(a, b, points)
    assert (got.ops, got.row_a, got.row_b) == (ops, ra, rb)


def test_local_end_cell_ties_every_path(ctx):
    """Two-letter sequences make many cells share the best local score; every kernel family must report
    the same one as the oracle (smallest i, then smallest j): packed short, packed long with 8 and with 16
    columns per lane, and the int32 single-pair tiles."""
    rng = np.random.default_rng(4242)
    ac = np.frombuffer(b"AC", dtype=np.uint8)

    def low_entropy(n):
        return ac[rng.integers(0, 2, size=n)].tobytes()

    for n_pairs, m_lo, m_hi, n_lo, n_hi in ((256, 100, 150, 100, 150), (64, 300, 600, 400, 900), (24, 900, 1100, 1030, 1400)):
        As = [low_entropy(int(rng.integers(m_lo, m_hi + 1))) for _ in range(n_pairs)]
        Bs = [low_entropy(int(rng.integers(n_lo, n_hi + 1))) for _ in range(n_pairs)]
        ba, oa, la = psa.pack_pairs(As)
        bb, ob, lb = psa.pack_pairs(Bs)
        items, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.LOCAL, 1, 2, traceback=False)
        for k in range(n_pairs):
            lin = po.score_linear(As[k], Bs[k], 1, 2, mode=psa.LOCAL)
            assert items[k]["score"] == lin.score, (n_pairs, k)
            assert (items[k]["end_i"], items[k]["end_j"]) == (lin.end_i, lin.end_j), (n_pairs, k, lin.score)
    for m, n in ((700, 1500), (1500, 1500), (300, 2600)):
        a, b = low_entropy(m), low_entropy(n)
        lin = po.score_linear(a, b, 1, 2, mode=psa.LOCAL)
        got = ctx.align_pair(a, b, psa.LOCAL, 1, 2, traceback=False)
        assert (got.score, got.end_i, got.end_j) == (lin.score, lin.end_i, lin.end_j), (m, n)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_traceback_ties_low_entropy(ctx, mode):
    """Predecessor ties (the reference's T1, T2, T3 equality order, subproblem_alignment.cpp:147-169) are
    rare on 4-letter random sequences and everywhere on 2-letter ones: full alignments against the oracle
    through the packed short kernels, the checkpointed long-pair traceback and its band tiles."""
    rng = np.random.default_rng(515 + mode)
    ac = np.frombuffer(b"AC", dtype=np.uint8)

    def low_entropy(n):
        return ac[rng.integers(0, 2, size=n)].tobytes()

    As = [low_entropy(int(rng.integers(60, 151))) for _ in range(192)]
    Bs = [low_entropy(int(rng.integers(60, 151))) for _ in range(192)]
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    for g, h in ((1, 2), (1, 1), (2, 0)):
        items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=True)
        for k in range(len(As)):
            w = po.align(As[k], Bs[k], g, h, mode=mode)
            assert items[k]["score"] == w.score and psa.unpack_ops(ops[k], int(items[k]["aln_len"])) == w.ops, (g, h, k)
            assert (items[k]["start_i"], items[k]["start_j"]) == (w.start_i, w.start_j), (g, h, k)
    for m, n in ((300, 700), (900, 1000), (1400, 1300)):
        a, b = low_entropy(m), low_entropy(n)
        w = po.align(a, b, 1, 2, mode=mode)
        got = ctx.align_pair(a, b, mode, 1, 2)
        assert got.score == w.score and got.ops == w.ops and (got.row_a, got.row_b) == (w.row_a, w.row_b), (m, n)


@pytest.mark.parametrize("geo", ["6", "7", "2", "0"])
def test_long_geometries_tie_prone(geo):
    """The wide-lane geometries the launcher only picks from ~485 kbp (24 columns per lane, 128- and 256-row
    blocks) forced onto small tie-prone pairs: score and end cell (local) / corner values (global) against
    the linear-space oracle."""
    ctx = psa.Context(0)
    ctx.set_option("long_geometry", int(geo))
    rng = np.random.default_rng(int(geo) + 900)
    ac = np.frombuffer(b"AC", dtype=np.uint8)
    for m, n in ((700, 1500), (1300, 2100), (257, 3000)):
        a = ac[rng.integers(0, 2, size=m)].tobytes()
        b = ac[rng.integers(0, 2, size=n)].tobytes()
        lin = po.score_linear(a, b, 1, 2, mode=psa.LOCAL)
        got = ctx.align_pair(a, b, psa.LOCAL, 1, 2, traceback=False)
        assert (got.score, got.end_i, got.end_j) == (lin.score, lin.end_i, lin.end_j), (geo, m, n)
        lin = po.score_linear(a, b, 1, 2, mode=psa.GLOBAL)
        got = ctx.align_pair(a, b, psa.GLOBAL, 1, 2, traceback=False)
        assert (got.t1, got.t2, got.t3, got.end_state) == (lin.t1, lin.t2, lin.t3, lin.end_state), (geo, m, n)
    ctx.close()


def _rescore_rows(row_a: bytes, row_b: bytes, g=1, h=2):
    score, prev = 0, 0
    for x, y in zip(row_a, row_b):
        t = 2 if x == 0x2D else (3 if y == 0x2D else 1)
        if t == 1:
            score += 1 if x == y else 0
        else:
            score -= g + (0 if t == prev else h)
        prev = t
    return score


@pytest.mark.parametrize("pieces", [2, 5, 16])
def test_partition_finder_stitched_alignment(ctx, pieces):
    """SURVEY 8 f-3 (the role of partial.cpp:81-163 + optimal_alignment): forward + reverse sweeps, best crossing per
    special row, typed pieces stitched.  The stitched alignment is complete (spells all of A and all of B), re-scores
    to the oracle's global optimum, and its crossings lie on the special rows -- on mutated copies, unrelated
    sequences, tie-prone two-letter sequences (many co-optimal paths) and a 13 kbp dataset pair."""
    rng = np.random.default_rng(400 + pieces)
    names, seqs = dataset()
    cases = []
    for (m, n) in ((1000, 1100), (3000, 2500), (129, 700), (2049, 300)):
        a = random_dna(rng, m)
        cases.append((a, mutated_copy(rng, a, n, ins=0.03, dele=0.03)))
    cases.append((random_dna(rng, 900), random_dna(rng, 1300)))
    ac = np.frombuffer(b"AC", dtype=np.uint8)
    cases.append((ac[rng.integers(0, 2, size=1500)].tobytes(), ac[rng.integers(0, 2, size=1400)].tobytes()))
    cases.append((b"A" * 700, b"A" * 900))
    cases.append((seqs[6][:13327].encode(), seqs[8][:13327].encode()))
    for a, b in cases:
        got, crossings = ctx.align_long_partitioned(a, b, pieces, 1, 2)
        lin = po.score_linear(a, b, 1, 2)
        assert got.score == lin.score, (len(a), len(b), pieces)
        assert got.row_a.replace(b"-", b"") == a and got.row_b.replace(b"-", b"") == b       # complete, in order
        assert _rescore_rows(got.row_a, got.row_b) == lin.score
        assert len(crossings) <= pieces - 1
        assert all(i % 128 == 0 and 0 < i < len(a) and 0 <= j <= len(b) and t in (1, 3) for i, j, t in crossings)
        assert crossings == sorted(crossings)
        if len(a) >= 1000 and pieces > 2:
            assert len(crossings) >= 1
