"""Batches of long pairs with traceback: the checkpointed one-warp-per-pair fill and the batched walk, through the
host entry (psa_align_batch), the device entry (psa_align_batch_device) and psa_align_partition, against the oracle's
full traceback and the per-pair path (align_pair, one pair over the whole GPU)."""
import random
import threading

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200 import synth
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE, PairResult
from oracle import pyoracle as po
from tests.helpers import mutated_copy, random_dna

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5A5A5A5


@pytest.fixture(scope="module")
def ctx():
    c = psa.Context(0)
    yield c
    c.close()


def _stride(As, Bs):
    return (max(map(len, As)) + max(map(len, Bs)) + 15) // 16 + 1


def _host(ctx, As, Bs, mode, g=1, h=2):
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    return ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=True)


def _device(ctx, As, Bs, mode, g=1, h=2, stride=None):
    """psa_align_batch_device on torch tensors, on a stream that is not the default one; the op buffer is filled with a
    sentinel first.  Returns (items, ops words [n, stride])."""
    import torch
    dev = torch.device("cuda", 0)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    n = len(As)
    stride = stride or _stride(As, Bs)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        pad = np.zeros(1, dtype=np.uint8)             # never an empty tensor, even when every member of one side is empty
        t = [torch.from_numpy(x).to(dev) for x in (np.concatenate([ba, pad]), oa, la, np.concatenate([bb, pad]), ob, lb)]
        items = torch.zeros(n * 10, dtype=torch.int32, device=dev)
        ops = torch.from_numpy(np.full(n * stride, SENTINEL, dtype=np.uint32).view(np.int32)).to(dev)
        st.synchronize()
        ctx.align_batch_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                               t[5].data_ptr(), n, int(la.max()), int(lb.max()), items.data_ptr(), ops.data_ptr(), stride,
                               mode, g, h, True, st.cuda_stream)
        st.synchronize()
    return items.cpu().numpy().view(ITEM_DTYPE).copy(), ops.cpu().numpy().view(np.uint32).reshape(n, stride).copy()


def _check(it, words, a, b, want, local, tag):
    """Whole-result comparison with an oracle alignment or a PairResult of align_pair (which carries t1..t3 in local mode
    too: then they are compared as well)."""
    assert it["score"] == want.score, tag
    if not local or isinstance(want, PairResult):
        assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (want.t1, want.t2, want.t3, want.end_state), tag
    assert (it["end_i"], it["end_j"]) == (want.end_i, want.end_j), tag
    assert (it["start_i"], it["start_j"]) == (want.start_i, want.start_j), tag
    n = int(it["aln_len"])
    ops = psa.unpack_ops(words, n)
    assert ops == want.ops, tag
    assert psa.render_rows(a, b, ops, int(it["start_i"]), int(it["start_j"])) == (want.row_a, want.row_b), tag


def _untouched_tail(words, it):
    used = (int(it["aln_len"]) + 15) // 16
    return bool((words[used:] == SENTINEL).all())


def _ragged(rng, count, lo=257, hi=2000):
    As, Bs = [], []
    for k in range(count):
        m = int(rng.integers(lo, hi + 1))
        n = int(rng.integers(lo, hi + 1))
        a = random_dna(rng, m)
        As.append(a)
        Bs.append(mutated_copy(rng, a, n) if k % 3 else random_dna(rng, n))     # m < n and m > n both occur
    return As, Bs


@pytest.mark.parametrize("gh", [(1, 2), (2, 1), (1, 0), (1, 5)])
@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_random_ragged_batches_both_entries(ctx, mode, gh):
    g, h = gh
    rng = np.random.default_rng(1000 + 10 * mode + g * 3 + h)
    As, Bs = _ragged(rng, 48)
    hi, ho = _host(ctx, As, Bs, mode, g, h)
    di, do = _device(ctx, As, Bs, mode, g, h)
    assert (hi == di).all()
    for k in range(len(As)):
        want = po.align(As[k], Bs[k], g, h, mode=mode)
        _check(hi[k], ho[k], As[k], Bs[k], want, mode == psa.LOCAL, k)
        _check(di[k], do[k], As[k], Bs[k], want, mode == psa.LOCAL, k)
        assert _untouched_tail(do[k], di[k]), k


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_tile_edges_in_one_batch(ctx, mode):
    rng = np.random.default_rng(77 + mode)
    As, Bs = [], []
    for m in (127, 128, 129):
        for n in (255, 256, 257, 511, 513):
            a = random_dna(rng, m)
            As.append(a)
            Bs.append(mutated_copy(rng, a, n) if (m + n) % 2 else random_dna(rng, n))
    items, ops = _host(ctx, As, Bs, mode)
    di, do = _device(ctx, As, Bs, mode)
    assert (items == di).all()
    for k in range(len(As)):
        _check(items[k], ops[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL, k)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_tie_prone_two_letter_sequences(ctx, mode):
    """Many co-optimal paths: predecessor order and end-cell ties must fall as the oracle's."""
    rng = np.random.default_rng(31 + mode)
    two = np.frombuffer(b"AC", dtype=np.uint8)
    As = [two[rng.integers(0, 2, size=int(rng.integers(300, 1300)))].tobytes() for _ in range(16)]
    Bs = [two[rng.integers(0, 2, size=int(rng.integers(300, 1300)))].tobytes() for _ in range(16)]
    items, ops = _host(ctx, As, Bs, mode)
    for k in range(len(As)):
        _check(items[k], ops[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL, k)


@pytest.mark.parametrize("n,period", [(700, 256), (1500, 512)])
def test_tie_prone_periodic_motifs(ctx, n, period):
    """The two-motif construction of the score-only tie test (two diagonals reach the same local score, the one at
    the smaller rows a strip further right), now with traceback through the batch path."""
    rng = np.random.default_rng(n + period)
    gt = np.frombuffer(b"GT", dtype=np.uint8)
    As, Bs = [], []
    for _ in range(24):
        m1 = gt[rng.integers(0, 2, size=48)].tobytes()
        m2 = gt[rng.integers(0, 2, size=48)].tobytes()
        a = bytearray(b"A" * 640)
        b = bytearray(b"C" * n)
        c1 = int(rng.integers(10, 150))
        r_big, r_small = 400 + int(rng.integers(0, 100)), 60 + int(rng.integers(0, 100))
        a[r_big:r_big + 48] = m1
        b[c1:c1 + 48] = m1
        a[r_small:r_small + 48] = m2
        b[c1 + period:c1 + period + 48] = m2
        As.append(bytes(a)); Bs.append(bytes(b))
    items, ops = _host(ctx, As, Bs, psa.LOCAL)
    ties = 0
    for k in range(len(As)):
        want = po.align(As[k], Bs[k], 1, 2, mode=po.LOCAL)
        _check(items[k], ops[k], As[k], Bs[k], want, True, k)
        ties += want.score == 48
    assert ties > 10


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_any_alphabet_and_empty_members(ctx, mode):
    """Non-ACGT bytes (N, bytes >= 128, NUL) and members with len_a == 0 or len_b == 0 inside a long batch: every member
    equals today's per-pair result (align_pair) and, where it has one, the oracle's."""
    rng = np.random.default_rng(5150 + mode)
    alpha = np.frombuffer(b"ACGTN\x80\xff\x00", dtype=np.uint8)
    As, Bs = [], []
    for k in range(12):
        a = alpha[rng.integers(0, len(alpha), size=int(rng.integers(257, 1200)))].tobytes()
        As.append(a)
        Bs.append(bytes(c if rng.random() > 0.1 else alpha[int(rng.integers(0, 8))] for c in a[:int(rng.integers(257, len(a) + 1))]))
    for (m, n) in ((0, 700), (900, 0), (0, 0), (0, 300)):
        As.append(random_dna(rng, m))
        Bs.append(random_dna(rng, n))
    pairs = list(zip(As, Bs))
    rng.shuffle(pairs)                        # the empty members end up between long ones
    As, Bs = [p[0] for p in pairs], [p[1] for p in pairs]
    assert sum(1 for a, b in pairs if not a or not b) >= 4
    hi, ho = _host(ctx, As, Bs, mode)
    di, do = _device(ctx, As, Bs, mode)
    assert (hi == di).all()
    for k in range(len(As)):
        one = ctx.align_pair(As[k], Bs[k], mode, 1, 2)
        _check(hi[k], ho[k], As[k], Bs[k], one, mode == psa.LOCAL, k)
        if As[k] and Bs[k]:
            _check(hi[k], ho[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL, k)
        else:
            assert hi[k]["aln_len"] == 0 and (do[k] == SENTINEL).all(), k


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_chunks_equal_one_chunk(mode):
    """A batch split into chunks of 5 pairs returns what one chunk returns and what the oracle returns, and no op
    word past a pair's own ceil(aln_len / 16) is written."""
    rng = np.random.default_rng(808 + mode)
    As, Bs = _ragged(rng, 23, 257, 1400)
    whole = psa.Context(0)
    split = psa.Context(0)
    split.set_option("long_tb_chunk", 5)
    try:
        wi, wo = _device(whole, As, Bs, mode)
        si, so = _device(split, As, Bs, mode)
        hi, ho = _host(split, As, Bs, mode)
    finally:
        whole.close()
        split.close()
    assert (wi == si).all() and (wo == so).all() and (hi == si).all()
    for k in range(len(As)):
        assert _untouched_tail(so[k], si[k]), k
        _check(si[k], so[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL, k)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_config5_shape_with_traceback(ctx, mode):
    """64 x 5 kbp pairs of the config-5 generator: equal pair by pair to align_pair (per-pair path), and to the oracle
    for a few of them."""
    A, B = synth.read_pair_batch(64, 5000, synth.SEED_C5)
    As = [A[k].tobytes() for k in range(64)]
    Bs = [B[k].tobytes() for k in range(64)]
    di, do = _device(ctx, As, Bs, mode)
    for k in range(64):
        _check(di[k], do[k], As[k], Bs[k], ctx.align_pair(As[k], Bs[k], mode, 1, 2), mode == psa.LOCAL, k)
    for k in (0, 1, 38):
        _check(di[k], do[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL, k)


def test_typed_wide_pieces_of_a_partition(ctx):
    """psa_align_partition with several pieces wider than 256 columns and arbitrary start / end types: the pieces run
    as one batch; linked result equal to oracle pieces linked the same way."""
    rng = np.random.default_rng(4242)
    for trial in range(6):
        m = int(rng.integers(5000, 7000))
        a = random_dna(rng, m)
        b = mutated_copy(rng, a, int(m + rng.integers(-40, 41)), sub=0.1, ins=0.03, dele=0.03)
        n = len(b)
        k = int(rng.integers(16, 21))             # 17 - 21 pieces: the batched path, not the per-pair loop
        ii = sorted(int(x) for x in rng.integers(0, m + 1, size=k))
        jj = sorted(int(x) for x in rng.integers(0, n + 1, size=k))
        types = [-3, -2, -1, 1, 2, 3]
        points = [(0, 0, -1)] + [(i, j, int(rng.choice(types))) for i, j in zip(ii, jj)] + [(m, n, 1)]
        ops = ra = rb = b""
        last = None
        for (i0, j0, t0), (i1, j1, t1) in zip(points[:-1], points[1:]):
            last = po.align(a[i0:i1], b[j0:j1], 1, 2, start_type=t0, end_type=-t1)
            ops += last.ops; ra += last.row_a; rb += last.row_b
        got = ctx.align_partition(a, b, points, 1, 2)
        assert (got.ops, got.row_a, got.row_b) == (ops, ra, rb), (trial, points)
        assert (got.t1, got.t2, got.t3, got.end_state) == (last.t1, last.t2, last.t3, last.end_state), trial


def test_threads_with_own_contexts():
    """8 host threads, one context each, long traceback batches of mixed shapes at the same time."""
    errors = []

    def work(t):
        try:
            c = psa.Context(0)
            rng = np.random.default_rng(9000 + t)
            for rep in range(2):
                lo, hi = [(257, 700), (600, 1800), (257, 1500)][(t + rep) % 3]
                As, Bs = _ragged(rng, 10 + t, lo, hi)
                mode = (t + rep) % 2
                items, ops = _host(c, As, Bs, mode) if rep == 0 else _device(c, As, Bs, mode)
                for k in range(len(As)):
                    _check(items[k], ops[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2, mode=mode), mode == psa.LOCAL,
                           (t, rep, k))
            c.close()
        except Exception as e:          # reported by the main thread
            errors.append((t, repr(e)))

    th = [threading.Thread(target=work, args=(t,)) for t in range(8)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors


def test_errors(ctx):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3)
    As, Bs = _ragged(rng, 6, 400, 600)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    t = [torch.from_numpy(x).to(dev) for x in (ba, oa, la, bb, ob, lb)]
    items = torch.zeros(6 * 10, dtype=torch.int32, device=dev)
    need = (int(la.max()) + int(lb.max()) + 15) // 16
    ops = torch.zeros(6 * need, dtype=torch.int32, device=dev)
    with pytest.raises(psa.PsaError) as e:
        ctx.align_batch_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                               t[5].data_ptr(), 6, int(la.max()), int(lb.max()), items.data_ptr(), ops.data_ptr(), need - 1,
                               psa.GLOBAL, 1, 2, True)
    assert e.value.code == -5                 # PSA_ERR_CAPACITY
    big = 2 ** 21 - 1
    with pytest.raises(psa.PsaError) as e:
        ctx.align_batch_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                               t[5].data_ptr(), 6, big, int(lb.max()), items.data_ptr(), ops.data_ptr(),
                               (big + int(lb.max()) + 15) // 16, psa.GLOBAL, 1, 2, True)
    assert e.value.code == -2                 # PSA_ERR_RANGE
    Al = [b"A" * big] + As[1:]
    with pytest.raises(psa.PsaError) as e:
        _host(ctx, Al, Bs, psa.LOCAL)
    assert e.value.code == -2
    torch.cuda.synchronize()
    # the context is still usable afterwards
    items_h, ops_h = _host(ctx, As, Bs, psa.GLOBAL)
    for k in range(len(As)):
        _check(items_h[k], ops_h[k], As[k], Bs[k], po.align(As[k], Bs[k], 1, 2), False, k)
