"""GPU parity of the short-pair kernel through the C-ABI against the oracle and the golden
vectors.  Bit-exact: corner values, end state, end/start cells, ops and printed rows."""
import hashlib
import json
import os
import random

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from oracle import pyoracle as po
from tests.helpers import GOLDEN, dataset, mutated_copy, py_random_pair, random_dna

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


def test_config1_pair(ctx):
    names, seqs = dataset()
    a, b = seqs[2][:50].encode(), seqs[15][:50].encode()
    got = ctx.align_pair(a, b)
    lines = open(os.path.join(GOLDEN, "g1_stdout.txt")).read().split("\n")
    assert got.row_a.decode() == lines[lines.index("bp4") + 1]
    assert got.row_b.decode() == lines[lines.index("bp4") + 2]
    assert (got.t1, got.t2, got.t3, got.end_state) == (9, 5, 7, 1)


def test_kat_fixtures(ctx):
    names, seqs = dataset()
    for case in json.load(open(os.path.join(GOLDEN, "kat.json"))):
        if "a" in case:
            a, b = case["a"].encode(), case["b"].encode()
        elif case["L"] <= 256:
            a, b = seqs[case["rec_a"]][:case["L"]].encode(), seqs[case["rec_b"]][:case["L"]].encode()
        else:
            continue
        got = ctx.align_pair(a, b, psa.GLOBAL, case["g"], case["h"])
        assert [got.t1, got.t2, got.t3] == case["corner"] and got.end_state == case["end_state"]
        assert hashlib.md5(got.row_a + b"\n" + got.row_b + b"\n").hexdigest() == case["md5"]


def test_random_small_fixture_batch(ctx):
    cases = json.load(open(os.path.join(GOLDEN, "random_small.json")))
    by_gh = {}
    for c in cases:
        by_gh.setdefault((c["g"], c["h"]), []).append(c)
    for (g, h), cs in by_gh.items():
        ba, oa, la = psa.pack_pairs([c["a"].encode() for c in cs])
        bb, ob, lb = psa.pack_pairs([c["b"].encode() for c in cs])
        items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.GLOBAL, g, h, traceback=True)
        for k, c in enumerate(cs):
            it = items[k]
            assert [it["t1"], it["t2"], it["t3"]] == c["corner"] and it["end_state"] == c["end_state"]
            fwd = psa.unpack_ops(ops[k], int(it["aln_len"]))
            ra, rb = psa.render_rows(c["a"].encode(), c["b"].encode(), fwd, int(it["start_i"]), int(it["start_j"]))
            assert (ra.decode(), rb.decode()) == (c["row_a"], c["row_b"])


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_random_pairs_vs_oracle(ctx, mode):
    rnd = random.Random(100 + mode)
    for t in range(300):
        a, b = py_random_pair(rnd, max_m=rnd.choice([8, 40, 130, 250]), max_n=rnd.choice([8, 48, 150, 256]),
                              alpha=rnd.choice([b"ACGT", b"AC", b"ACGTN"]))
        b = b[:256]
        g, h = rnd.choice([(1, 2), (1, 2), (2, 1), (1, 0), (0, 3), (3, 5)])
        got = ctx.align_pair(a, b, mode, g, h)
        want = po.align(a, b, g, h, mode=mode)
        _same(got, want, local=(mode == psa.LOCAL))


def test_m_greater_than_n_and_edges(ctx):
    # outside the reference's m <= n contract the library still follows the oracle
    for a, b in [(b"ACGTACGTAC", b"ACG"), (b"A", b"A"), (b"A", b"C"), (b"AAAA", b"A" * 200), (b"", b"ACG"),
                 (b"ACG", b""), (b"", b"")]:
        for mode in (psa.GLOBAL, psa.LOCAL):
            got = ctx.align_pair(a, b, mode, 1, 2)
            if len(a) and len(b):
                _same(got, po.align(a, b, 1, 2, mode=mode), local=(mode == psa.LOCAL))
            else:
                assert got.ops == b"" and got.row_a == b""
                if mode == psa.GLOBAL:
                    lin = po.score_linear(a, b, 1, 2)
                    assert (got.t1, got.t2, got.t3) == (lin.t1, lin.t2, lin.t3)


def test_config2_slice_local(ctx):
    """BASELINE config 2 shape: 150 bp x 150 bp, even pairs mutated copies, odd pairs random."""
    rng = np.random.default_rng(20250002)
    n = 2048
    As = [random_dna(rng, 150) for _ in range(n)]
    Bs = [mutated_copy(rng, x, 150) if k % 2 == 0 else random_dna(rng, 150) for k, x in enumerate(As)]
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.LOCAL, 1, 2, traceback=True)
    lin = po.score_batch(ba, oa, la, bb, ob, lb, 1, 2, mode=po.LOCAL)
    for k in range(n):
        assert (items[k]["score"], items[k]["end_i"], items[k]["end_j"]) == (lin[k].score, lin[k].end_i, lin[k].end_j)
    for k in range(0, n, 8):
        w = po.align(As[k], Bs[k], 1, 2, mode=po.LOCAL)
        assert psa.unpack_ops(ops[k], int(items[k]["aln_len"])) == w.ops
        assert (items[k]["start_i"], items[k]["start_j"]) == (w.start_i, w.start_j)
    # score-only path agrees with the traceback path
    items2, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.LOCAL, 1, 2, traceback=False)
    assert np.array_equal(items2["score"], items["score"]) and np.array_equal(items2["end_j"], items["end_j"])


def test_error_codes(ctx):
    with pytest.raises(psa.PsaError) as e:
        ctx.align_pair(b"ACGT", b"ACGT", psa.GLOBAL, -1, 2)
    assert e.value.code == -1


@pytest.mark.parametrize("g,h,mode,max_m,max_n", [(1, 2, psa.GLOBAL, 40, 48), (1, 2, psa.GLOBAL, 96, 128),
                                                  (1, 2, psa.LOCAL, 96, 128), (2, 1, psa.GLOBAL, 150, 150),
                                                  (0, 2, psa.GLOBAL, 30, 30), (1, 0, psa.LOCAL, 200, 256),
                                                  (1, 2, psa.LOCAL, 150, 150), (1, 1, psa.GLOBAL, 300, 180),
                                                  (1, 2, psa.LOCAL, 90, 96), (1, 2, psa.GLOBAL, 100, 160),
                                                  (2, 2, psa.LOCAL, 17, 20)])
@pytest.mark.parametrize("flavour", [0, 1])
def test_packed_kernel_ragged_batches(g, h, mode, max_m, max_n, flavour):
    """The .S16x2 kernel (two pairs per register, >= 64 pairs per call): ragged lengths, members
    with other alphabets / lower case / zero length mixed in (those take the generic kernel).  Both
    traceback flavours: direction-code ring (0) and tile-boundary checkpoints + per-tile recompute (1)."""
    ctx = psa.Context(0)
    ctx.set_option("pack_traceback", flavour)
    rnd = random.Random(g * 1000 + h * 100 + mode * 10 + max_m)
    pairs = []
    for k in range(160):
        a, b = py_random_pair(rnd, max_m, max_n, b"ACGT")
        b = b[:max_n]
        if k % 23 == 5:
            a, b = a.replace(b"A", b"N"), b
        if k % 29 == 7:
            b = b.lower()
        if k % 31 == 9:
            a = b""
        if k % 37 == 11:
            a, b = py_random_pair(rnd, max_m, max_n, b"ABCDEFGHIJKLMNOPQRSTUVWY")
            b = b[:max_n]
        pairs.append((a, b))
    ba, oa, la = psa.pack_pairs([a for a, b in pairs])
    bb, ob, lb = psa.pack_pairs([b for a, b in pairs])
    for tb in (True, False):
        items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=tb)
        for k, (a, b) in enumerate(pairs):
            it = items[k]
            if len(a) == 0 or len(b) == 0:
                assert it["aln_len"] == 0
                continue
            w = po.align(a, b, g, h, mode=mode)
            assert it["score"] == w.score and (it["end_i"], it["end_j"]) == (w.end_i, w.end_j), k
            if mode == psa.GLOBAL:
                assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (w.t1, w.t2, w.t3, w.end_state), k
            if tb:
                assert psa.unpack_ops(ops[k], int(it["aln_len"])) == w.ops, k
                assert (it["start_i"], it["start_j"]) == (w.start_i, w.start_j), k
    ctx.close()


def test_concurrent_host_threads_like_the_harness():
    """The reference harness calls the boundary function from hardware_concurrency() host threads at
    once (testing.cpp:145-152).  One context per thread, all threads aligning their own pairs."""
    import threading
    rnd = random.Random(99)
    jobs = [py_random_pair(rnd, 120, 200, b"ACGT") for _ in range(64)]
    jobs = [(a, b[:200]) for a, b in jobs]
    want = [po.align(a, b, 1, 2) for a, b in jobs]
    got = [None] * len(jobs)
    errors = []

    def worker(t, nthreads):
        try:
            c = psa.Context(0)
            for k in range(t, len(jobs), nthreads):
                got[k] = c.align_pair(jobs[k][0], jobs[k][1], psa.GLOBAL, 1, 2)
            c.close()
        except Exception as e:  # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(t, 8)) for t in range(8)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    for g, w in zip(got, want):
        _same(g, w)


def test_capacity_and_range_errors(ctx):
    a, b = b"ACGT" * 30, b"ACGT" * 30
    ba, oa, la = psa.pack_pairs([a])
    bb, ob, lb = psa.pack_pairs([b])
    items = np.zeros(1, dtype=psa.capi.ITEM_DTYPE)
    ops = np.zeros((1, 2), dtype=np.uint32)          # far too small for 240 ops
    with pytest.raises(psa.PsaError) as e:
        ctx.align_batch(ba, oa, la, bb, ob, lb, psa.GLOBAL, 1, 2, traceback=True, items=items, ops=ops)
    assert e.value.code == -5                        # PSA_ERR_CAPACITY
    with pytest.raises(psa.PsaError) as e:
        ctx.align_pair(a, b, 7, 1, 2)                # unknown mode
    assert e.value.code == -1
    with pytest.raises(psa.PsaError) as e:
        ctx.align_pair(a, b, psa.GLOBAL, 10_000_000, 2)   # score range beyond int32 lanes
    assert e.value.code == -2


def test_size_limits_of_each_path(ctx):
    """Pairs at the edges of the kernels' envelopes: packed kernel maxima (m=512, n=256), the generic
    shared-memory kernel with tall pairs (m=1500), and the hand-over to the long path (n=257)."""
    rng = np.random.default_rng(2024)
    cases = [(512, 256), (511, 255), (1500, 200), (1700, 33), (1, 256), (256, 1), (700, 257)]
    for mode in (psa.GLOBAL, psa.LOCAL):
        for (m, n) in cases:
            a = random_dna(rng, m)
            b = mutated_copy(rng, a, n) if m >= n else mutated_copy(rng, a + random_dna(rng, n - m), n)
            _same(ctx.align_pair(a, b, mode, 1, 2), po.align(a, b, 1, 2, mode=mode), local=(mode == psa.LOCAL))
    # a batch at the packed kernel's maxima (>= 64 pairs so that it takes the .S16x2 path)
    As = [random_dna(rng, 512 - (k % 5)) for k in range(72)]
    Bs = [mutated_copy(rng, x, 256 - (k % 3)) for k, x in enumerate(As)]
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    for mode in (psa.GLOBAL, psa.LOCAL):
        items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=True)
        for k in range(0, 72, 7):
            w = po.align(As[k], Bs[k], 1, 2, mode=mode)
            assert items[k]["score"] == w.score and psa.unpack_ops(ops[k], int(items[k]["aln_len"])) == w.ops


def test_typed_subproblems_fixture_and_random(ctx):
    """SURVEY 8 f-2: the other border variants of Subproblem (start/end types), against the answers
    recorded from the reference and against the oracle on larger random pairs."""
    for case in json.load(open(os.path.join(GOLDEN, "typed_small.json"))):
        got = ctx.align_pair(case["a"].encode(), case["b"].encode(), psa.GLOBAL, case["g"], case["h"],
                             start_type=case["start_type"], end_type=case["end_type"])
        assert [got.t1, got.t2, got.t3] == case["corner"] and got.end_state == case["end_state"], case
        assert got.row_a.decode() == case["row_a"] and got.row_b.decode() == case["row_b"], case
    rng = np.random.default_rng(77)
    for st in (-1, -2, -3, 1, 2, 3):
        for et in (-1, -2, -3, 1, 2, 3):
            for t in range(4):
                m = int(rng.integers(1, 300))
                n = int(rng.integers(1, 257))
                a = random_dna(rng, m)
                b = mutated_copy(rng, a, n) if t % 2 else random_dna(rng, n)
                g, h = [(1, 2), (2, 1), (1, 0), (0, 3)][int(rng.integers(0, 4))]
                want = po.align(a, b, g, h, start_type=st, end_type=et)
                _same(ctx.align_pair(a, b, psa.GLOBAL, g, h, start_type=st, end_type=et), want)
    a, b = random_dna(rng, 400), random_dna(rng, 400)      # wider than the short kernel takes: long-pair kernels
    _same(ctx.align_pair(a, b, start_type=2, end_type=-3), po.align(a, b, 1, 2, start_type=2, end_type=-3))
    with pytest.raises(psa.PsaError) as e:
        ctx.align_pair(b"ACGT", b"ACGT", start_type=4)
    assert e.value.code == -1


def _oracle_partition(a, b, points, g, h):
    """The intended optimal_alignment (main_alignment.cpp:202-350) from oracle pieces: piece k from
    point k to point k+1, start type t_k, end type -t_{k+1}, alignments linked in order."""
    ops, ra, rb = b"", b"", b""
    last = None
    for (i0, j0, t0), (i1, j1, t1) in zip(points[:-1], points[1:]):
        last = po.align(a[i0:i1], b[j0:j1], g, h, start_type=t0, end_type=-t1)
        ops += last.ops; ra += last.row_a; rb += last.row_b
    return ops, ra, rb, last


def test_partitioned_alignment(ctx):
    rng = np.random.default_rng(2025)
    for trial in range(40):
        m = int(rng.integers(30, 900))
        a = random_dna(rng, m)
        b = mutated_copy(rng, a, int(m + rng.integers(-20, 21)), sub=0.1, ins=0.03, dele=0.03)
        n = len(b)
        g, h = [(1, 2), (2, 1), (1, 0)][trial % 3]
        if trial % 2 == 0:
            # points on an optimal path of the whole problem: nodes of the oracle's own alignment
            whole = po.align(a, b, g, h)
            i, j = whole.start_i, whole.start_j
            nodes = []
            for k, t in enumerate(whole.ops):
                if k:
                    i += t != 2; j += t != 3
                nodes.append((i, j, t))
            picks = sorted(set(int(x) for x in rng.integers(0, len(nodes), size=int(rng.integers(1, 8)))))
            points = [(0, 0, -1)] + [nodes[k] for k in picks if 0 < nodes[k][0] < m and 0 < nodes[k][1] < n] + [(m, n, 1)]
        else:
            # arbitrary monotone points with arbitrary types (including empty pieces)
            k = int(rng.integers(1, 10))
            ii = sorted(int(x) for x in rng.integers(0, m + 1, size=k))
            jj = sorted(int(x) for x in rng.integers(0, n + 1, size=k))
            points = [(0, 0, -1)] + [(i, j, int(rng.choice([-3, -2, -1, 1, 2, 3]))) for i, j in zip(ii, jj)] + [(m, n, 1)]
        ops, ra, rb, last = _oracle_partition(a, b, points, g, h)
        got = ctx.align_partition(a, b, points, g, h)
        assert (got.ops, got.row_a, got.row_b) == (ops, ra, rb), (trial, points)
        assert (got.t1, got.t2, got.t3, got.end_state) == (last.t1, last.t2, last.t3, last.end_state)
    # the live configuration: two points = the single subproblem (main_alignment.cpp:392-398)
    a, b = b"GATTACAGATTACA", b"GATCACAGGATTAA"
    one = ctx.align_pair(a, b)
    two = ctx.align_partition(a, b, [(0, 0, -1), (len(a), len(b), 1)])
    assert (one.ops, one.row_a, one.row_b) == (two.ops, two.row_a, two.row_b)
    with pytest.raises(psa.PsaError):
        ctx.align_partition(a, b, [(0, 0, -1), (5, 5, 1), (4, 8, 1)])      # decreasing
    with pytest.raises(psa.PsaError):
        ctx.align_partition(a, b, [(0, 0, -1)])


def test_sequence_similarity_batch(ctx):
    """SURVEY 8 f-4: sequence_similarity (pull_data.cpp:97-127) on the GPU against numpy, with ragged
    lengths (every alignment of the two byte streams), empty members and long records."""
    rng = np.random.default_rng(11)
    seqs_a, seqs_b = [], []
    for k in range(700):
        la = int(rng.integers(0, 40)) if k % 3 else int(rng.integers(0, 700))
        lb = int(rng.integers(0, 40)) if k % 5 else int(rng.integers(0, 700))
        a = random_dna(rng, la)
        b = mutated_copy(rng, a, lb, sub=0.2) if k % 2 else random_dna(rng, lb)
        seqs_a.append(a); seqs_b.append(b)
    names, seqs = dataset()
    seqs_a += [seqs[2].encode(), seqs[0].encode(), b"", b"ACGT"]
    seqs_b += [seqs[15].encode(), seqs[1].encode()[:9000], b"ACGT", b""]
    ba, oa, la = psa.pack_pairs(seqs_a)
    bb, ob, lb = psa.pack_pairs(seqs_b)
    got = ctx.similarity_batch(ba, oa, la, bb, ob, lb)
    for k, (a, b) in enumerate(zip(seqs_a, seqs_b)):
        n = min(len(a), len(b))
        eq = int(np.count_nonzero(np.frombuffer(a[:n], dtype=np.uint8) == np.frombuffer(b[:n], dtype=np.uint8)))
        want = eq / max(len(a), len(b)) if max(len(a), len(b)) else 0.0
        assert got[k] == want, (k, len(a), len(b), got[k], want)


@pytest.mark.parametrize("mode", [psa.LOCAL, psa.GLOBAL])
@pytest.mark.parametrize("shape", [(150, 150), (97, 130), (33, 17), (300, 250)])
def test_packed_2bit_batch_equals_oracle_and_byte_api(ctx, mode, shape):
    """psa_align_batch_packed (fixed-stride 2-bit reads, 16-byte records): same scores, cells and ops as the
    oracle and as psa_align_batch on the unpacked reads; with and without traceback; through the chunked pipeline
    (n > chunk) as well."""
    from cse305_parallel_sequence_alignment_b200 import synth
    m, n_ = shape
    npairs = 3000
    A, _ = synth.read_pair_batch(npairs, m, 77 + m)
    rng = np.random.default_rng(5 + n_)
    B = synth.ACGT[synth.random_codes(rng, npairs, n_)]
    k = min(m, n_)
    B[0::2, :k] = A[0::2, :k]                              # even pairs share a prefix, with a few substitutions
    mut = rng.random((npairs, n_)) < 0.06
    B[mut] = synth.ACGT[rng.integers(0, 4, size=int(mut.sum()))]
    a2, b2 = psa.pack_reads_2bit(A), psa.pack_reads_2bit(B)
    c = psa.Context(0)
    c.set_option("pack_chunk", 1024)                       # 3000 pairs -> several chunks + ramps
    for tb in (True, False, "ckpt"):
        if tb == "ckpt":                                   # the checkpoint + tile-recompute traceback reads 2-bit input too
            c.set_option("pack_traceback", 1)
            tb = True
        items, ops = c.align_batch_packed(a2, b2, m, n_, mode, 1, 2, traceback=tb)
        offa, la = synth.fixed_length_layout(npairs, m)
        offb, lb = synth.fixed_length_layout(npairs, n_)
        ref_items, ref_ops = ctx.align_batch(A.reshape(-1), offa, la, B.reshape(-1), offb, lb, mode, 1, 2, traceback=tb)
        for f in ("score", "end_i", "end_j", "end_state") + (("start_i", "start_j", "aln_len") if tb else ()):
            assert np.array_equal(items[f].astype(np.int64), ref_items[f].astype(np.int64)), (f, tb)
        for q in range(0, npairs, 97):
            w = po.align(A[q].tobytes(), B[q].tobytes(), 1, 2, mode=mode)
            assert (items[q]["score"], items[q]["end_i"], items[q]["end_j"]) == (w.score, w.end_i, w.end_j)
            if tb:
                assert psa.unpack_ops(ops[q], int(items[q]["aln_len"])) == w.ops
                assert psa.unpack_ops(ref_ops[q], int(ref_items[q]["aln_len"])) == w.ops
    c.close()


@pytest.mark.parametrize("pinned, serial", [pytest.param(False, 0, id="False"), pytest.param(True, 0, id="True"),
                                            pytest.param(True, 1, id="True-serial_fills")])
def test_packed_2bit_compact_ops(ctx, pinned, serial):
    """PSA_OPS_COMPACT: op words back to back in pair order (page-locked and pageable
    destination) hold exactly the words of the fixed-stride layout; several chunks, ramps, empty alignments;
    fills of consecutive chunks concurrent or serialised (pack_serial_fills)."""
    import torch
    from cse305_parallel_sequence_alignment_b200 import synth
    npairs, L = 5000, 150
    A, B = synth.read_pair_batch(npairs, L, 4242)
    B[7] = synth.ACGT[(np.searchsorted(synth.ACGT, A[7]) + 2) % 4]       # no base in common position-wise; alignment may be tiny
    a2, b2 = psa.pack_reads_2bit(A), psa.pack_reads_2bit(B)
    c = psa.Context(0)
    c.set_option("pack_chunk", 1024)
    c.set_option("pack_serial_fills", serial)
    items, ops = c.align_batch_packed(a2, b2, L, L, psa.LOCAL, 1, 2, traceback=True)
    stride = ops.shape[1]
    if pinned:
        buf = torch.zeros(npairs * stride, dtype=torch.int32).pin_memory().numpy().view(np.uint32).reshape(npairs, stride)
    else:
        buf = np.zeros((npairs, stride), dtype=np.uint32)
    buf[:] = 0xDEADBEEF
    items_c, cops = c.align_batch_packed(a2, b2, L, L, psa.LOCAL, 1, 2, traceback=True, ops=buf, compact=True)
    assert np.array_equal(items_c, items)
    off = psa.compact_ops_offsets(items_c)
    flat = cops.reshape(-1)
    for k in range(npairs):
        w = int(off[k + 1] - off[k])
        assert w == (int(items[k]["aln_len"]) + 15) // 16
        assert np.array_equal(flat[off[k]:off[k + 1]], ops[k, :w]), k
    assert flat[off[-1]] == 0xDEADBEEF                 # nothing written past the last pair's words
    c.close()


def test_packed_2bit_batch_errors(ctx):
    a2 = np.zeros((4, 40), dtype=np.uint32)
    with pytest.raises(psa.PsaError) as e:
        ctx.align_batch_packed(a2, a2, 600, 600, psa.LOCAL, 1, 2)       # beyond the short-read envelope
    assert e.value.code == -2
    with pytest.raises(psa.PsaError) as e:
        small = np.ascontiguousarray(a2[:, :10])
        ctx.align_batch_packed(small, small, 150, 150, psa.LOCAL, 1, 5)   # h > 2: int32 kernels only
    assert e.value.code == -2
