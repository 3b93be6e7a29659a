"""Banded batches (psa_align_batch_banded, psa_align_batch_banded_device): the score-only <128, 16> grid and the
checkpointed <128, 8> traceback grid against the banded oracle, against psa_align_batch when the band holds every
cell, and at scale against the linear-space banded oracle."""
import random
import threading

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200 import synth
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE, NEG_INF, PsaError
from oracle import pyoracle as po
from tests import banded_oracle as bo
from tests.helpers import mutated_copy, random_dna

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5A5A5A5
FIELDS = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j")
NARROW = [0, 1, 7, 31, 32, 127, 128, 255, 256, 300]


@pytest.fixture(scope="module")
def ctx():
    c = psa.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_chunked():
    c = psa.Context(0)
    c.set_option("long_tb_chunk", 3)
    yield c
    c.close()


def _stride(As, Bs):
    return (max(map(len, As)) + max(map(len, Bs)) + 15) // 16 + 1


def _host(ctx, As, Bs, band, mode, g=1, h=2, tb=True):
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    return ctx.align_batch_banded(ba, oa, la, bb, ob, lb, band, mode, g, h, traceback=tb)


def _device(ctx, As, Bs, band, mode, g=1, h=2, tb=True, stride=None):
    """The device entry on torch tensors and a side stream; the op buffer starts as a sentinel."""
    import torch
    dev = torch.device("cuda", 0)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    n = len(As)
    stride = stride or _stride(As, Bs)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        pad = np.zeros(1, dtype=np.uint8)
        t = [torch.from_numpy(x).to(dev) for x in (np.concatenate([ba, pad]), oa, la, np.concatenate([bb, pad]), ob, lb)]
        items = torch.zeros(n * 10, dtype=torch.int32, device=dev)
        ops = torch.from_numpy(np.full(n * stride, SENTINEL, dtype=np.uint32).view(np.int32)).to(dev)
        st.synchronize()
        ctx.align_batch_banded_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                                      t[5].data_ptr(), n, int(la.max()), int(lb.max()), band, items.data_ptr(),
                                      ops.data_ptr() if tb else 0, stride if tb else 0, mode, g, h, tb, st.cuda_stream)
        st.synchronize()
    return items.cpu().numpy().view(ITEM_DTYPE).copy(), ops.cpu().numpy().view(np.uint32).reshape(n, stride).copy()


def rescore(a, b, ops, start_i, start_j, g, h, mode):
    """Score of the emitted columns plus, in global mode, the border run the traceback stops at."""
    if ops and mode == psa.GLOBAL:
        t = ops[0]
        pi, pj = start_i - (t != 2), start_j - (t != 3)
        ops = bytes([3] * pi if pj == 0 else [2] * pj) + ops
        i = j = 0
    else:
        i, j = start_i - 1, start_j - 1
    sc, prev = 0, 0
    for t in ops:
        if t == 1:
            sc += a[i] == b[j]
            i += 1
            j += 1
        else:
            sc -= (0 if t == prev else h) + g
            i += t == 3
            j += t == 2
        prev = t
    return sc


def in_band(a, b, ops, start_i, start_j, band):
    m, n = len(a), len(b)
    i, j = start_i, start_j
    for k, t in enumerate(ops):
        if k:
            i += t != 2
            j += t != 3
        if abs(j - i * n // m) > band:
            return False
    return True


def check_oracle(As, Bs, items, ops, band, mode, g=1, h=2, tb=True, tag=""):
    for k, (a, b) in enumerate(zip(As, Bs)):
        w = bo.align_banded(a, b, band, g, h, mode)
        it = items[k]
        assert tuple(int(it[f]) for f in FIELDS) == tuple(getattr(w, f) for f in FIELDS), (tag, k, len(a), len(b), band, it, w)
        if not tb:
            assert int(it["aln_len"]) == 0
            continue
        assert (int(it["start_i"]), int(it["start_j"]), int(it["aln_len"])) == (w.start_i, w.start_j, len(w.ops)), (tag, k, it, w)
        got = psa.unpack_ops(ops[k], int(it["aln_len"]))
        assert got == w.ops, (tag, k, band)
        if w.score != po.NEG and len(a) and len(b):
            assert rescore(a, b, got, w.start_i, w.start_j, g, h, mode) == w.score, (tag, k)


def _narrow_cases(rng, rnd):
    As, Bs = [], []
    for m, n in [(300, 300), (1000, 1000), (900, 120), (120, 900), (513, 257), (256, 256), (257, 512), (129, 700),
                 (1, 1000), (1000, 1), (0, 40), (40, 0), (128, 128)]:
        a = random_dna(rng, m)
        As.append(a)
        Bs.append(mutated_copy(rng, a, n) if m and n and rnd.random() < 0.7 else random_dna(rng, n))
    As.append(bytes(rnd.randrange(256) for _ in range(400)))            # any alphabet
    Bs.append(bytes(rnd.randrange(256) for _ in range(380)))
    return As, Bs


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_wide_band_equals_align_batch(ctx, mode):
    rng = np.random.default_rng(5100 + mode)
    As = [random_dna(rng, int(rng.integers(257, 2001))) for _ in range(12)]
    Bs = [mutated_copy(rng, a, int(rng.integers(257, 2001))) if k % 2 else random_dna(rng, int(rng.integers(257, 2001)))
          for k, a in enumerate(As)]
    As.append(b"")
    Bs.append(b"ACGT")
    band = max(map(len, As + Bs))
    for g, h in [(1, 2), (0, 0), (0, 1), (2, 0), (3, 1), (5, 2)]:
        ba, oa, la = psa.pack_pairs(As)
        bb, ob, lb = psa.pack_pairs(Bs)
        ref_items, ref_ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=True)
        for items, ops in (_host(ctx, As, Bs, band, mode, g, h), _device(ctx, As, Bs, band + 5, mode, g, h)):
            assert items.tobytes() == ref_items.tobytes(), (g, h)
            for k in range(len(As)):
                L = (int(items[k]["aln_len"]) + 15) // 16
                assert np.array_equal(ops[k, :L], ref_ops[k, :L]), (g, h, k)
        ref_s, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=False)
        items, _ = _host(ctx, As, Bs, band, mode, g, h, tb=False)
        assert items.tobytes() == ref_s.tobytes(), (g, h)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_narrow_bands_match_banded_oracle(ctx, mode):
    rng = np.random.default_rng(5200 + mode)
    rnd = random.Random(5201 + mode)
    As, Bs = _narrow_cases(rng, rnd)
    for band in NARROW:
        items, ops = _device(ctx, As, Bs, band, mode)
        check_oracle(As, Bs, items, ops, band, mode, tag=f"device tb {band}")
        for k, it in enumerate(items):          # no path / empty members: the op words stay untouched
            if int(it["aln_len"]) == 0:
                assert (ops[k] == SENTINEL).all(), (band, k)
        hitems, _ = _host(ctx, As, Bs, band, mode)
        assert hitems.tobytes() == items.tobytes(), band
        # score-only grid (K = 16) admits the same cells as the traceback grid (K = 8)
        sitems, _ = _host(ctx, As, Bs, band, mode, tb=False)
        check_oracle(As, Bs, sitems, None, band, mode, tb=False, tag=f"score {band}")
        ditems, _ = _device(ctx, As, Bs, band, mode, tb=False)
        assert ditems.tobytes() == sitems.tobytes(), band
        for f in FIELDS:
            assert np.array_equal(sitems[f], items[f]), (band, f)


def test_no_global_path(ctx):
    # n > (2*band + 1) * m leaves gaps between the band rows; with n <= m c(i) rises by at most 1 per row and a path
    # always exists (the 1000 x 1 pair: every cell is in the band)
    As, Bs = [b"A", b"AC", b"ACGTACGTAC", b"ACGT" * 250], [b"ACGT" * 250, b"ACGT" * 250, b"ACGTACGTAC", b"A"]
    items, ops = _device(ctx, As, Bs, 10, psa.GLOBAL)
    for k in range(2):
        it = items[k]
        assert (int(it["t1"]), int(it["t2"]), int(it["t3"]), int(it["score"]), int(it["end_state"]), int(it["aln_len"])) == \
               (NEG_INF, NEG_INF, NEG_INF, NEG_INF, 1, 0)
        assert (ops[k] == SENTINEL).all()
    assert int(items[2]["score"]) == 10 and int(items[3]["score"]) > NEG_INF
    check_oracle(As, Bs, items, ops, 10, psa.GLOBAL)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_tie_prone_sequences(ctx, mode):
    rnd = random.Random(5300 + mode)
    As, Bs = [], []
    for _ in range(6):
        m, n = rnd.randint(200, 900), rnd.randint(200, 900)
        As.append(bytes(rnd.choice(b"AB") for _ in range(m)))
        Bs.append(bytes(rnd.choice(b"AB") for _ in range(n)))
    for motif in (b"AC", b"ACG", b"AACG"):
        As.append(motif * (700 // len(motif)))
        Bs.append(motif * (650 // len(motif)) + b"T")
    for band in (0, 7, 32, 128, 257):
        for g, h in ((1, 2), (0, 1), (2, 0)):
            items, ops = _host(ctx, As, Bs, band, mode, g, h)
            check_oracle(As, Bs, items, ops, band, mode, g, h, tag=f"ties {band} {g} {h}")


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_chunked_equals_one_chunk(ctx, ctx_chunked, mode):
    rng = np.random.default_rng(5400 + mode)
    As = [random_dna(rng, int(rng.integers(300, 1500))) for _ in range(10)]
    Bs = [mutated_copy(rng, a, int(rng.integers(300, 1500))) for a in As]
    for band in (31, 256):
        one = _device(ctx, As, Bs, band, mode)
        many = _device(ctx_chunked, As, Bs, band, mode)
        assert one[0].tobytes() == many[0].tobytes() and np.array_equal(one[1], many[1]), band
        check_oracle(As, Bs, one[0], one[1], band, mode)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_100kbp_prefix_against_linear_banded_oracle(ctx, mode):
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    a, b = A[:100_000].tobytes(), B[:100_000].tobytes()
    want = bo.score_banded(a, b, 2000, 1, 2, mode)
    for tb in (False, True):
        items, _ = _host(ctx, [a], [b], 2000, mode, tb=tb)
        it = items[0]
        assert tuple(int(it[f]) for f in FIELDS) == (want.t1, want.t2, want.t3, want.score, want.end_state, want.end_i,
                                                     want.end_j), (tb, it)


def test_1Mbp_traceback_in_one_call_with_band_sized_memory():
    import torch
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    a, b = A.tobytes(), B.tobytes()
    torch.cuda.init()
    free0, _ = torch.cuda.mem_get_info()
    c = psa.Context(0)
    items, ops = _host(c, [a], [b], 1000, psa.GLOBAL)
    free1, _ = torch.cuda.mem_get_info()
    c.close()
    used = free0 - free1
    print(f"1 Mbp banded traceback: context allocated {used / 2**30:.2f} GiB")
    assert used < 2 * 2**30, used              # band-sized: the unbanded checkpoints would take ~94 GB
    it = items[0]
    assert int(it["score"]) > 0 and int(it["aln_len"]) >= 1_000_000
    got = psa.unpack_ops(ops[0], int(it["aln_len"]))
    assert rescore(a, b, got, int(it["start_i"]), int(it["start_j"]), 1, 2, psa.GLOBAL) == int(it["score"])
    assert in_band(a, b, got, int(it["start_i"]), int(it["start_j"]), 1000)


def test_errors(ctx):
    As, Bs = [b"ACGT" * 100], [b"ACGA" * 100]
    with pytest.raises(PsaError) as e:
        _host(ctx, As, Bs, -1, psa.GLOBAL)
    assert e.value.code == -1
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    with pytest.raises(PsaError) as e:
        ctx.align_batch_banded(ba, oa, la, bb, ob, lb, 10, psa.GLOBAL, flags=psa.WANT_SCORE | psa.OPS_COMPACT, traceback=False)
    assert e.value.code == -1
    big = b"A" * (2 ** 21 - 1)
    with pytest.raises(PsaError) as e:
        _host(ctx, [big], [b"ACGT"], 10, psa.GLOBAL, tb=False)
    assert e.value.code == -2
    with pytest.raises(PsaError) as e:
        ctx.align_batch_banded(ba, oa, la, bb, ob, lb, 10, psa.GLOBAL, ops=np.zeros((1, 49), dtype=np.uint32))
    assert e.value.code == -5
    with pytest.raises(PsaError) as e:
        _device(ctx, As, Bs, 10, psa.GLOBAL, stride=49)
    assert e.value.code == -5
    with pytest.raises(PsaError) as e:
        _device(ctx, As, Bs, -3, psa.LOCAL)
    assert e.value.code == -1


def test_threads_mix_banded_and_unbanded():
    errors = []

    def work(t):
        try:
            c = psa.Context(0)
            rng = np.random.default_rng(5500 + t)
            mode = psa.LOCAL if t % 2 else psa.GLOBAL
            for it_ in range(3):
                As = [random_dna(rng, int(rng.integers(200, 700))) for _ in range(5)]
                Bs = [mutated_copy(rng, a, int(rng.integers(200, 700))) for a in As]
                band = (7, 64, 300)[it_]
                items, ops = _host(c, As, Bs, band, mode)
                check_oracle(As, Bs, items, ops, band, mode)
                ba, oa, la = psa.pack_pairs(As)
                bb, ob, lb = psa.pack_pairs(Bs)
                ui, uo = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=True)
                for k in range(len(As)):
                    w = po.align(As[k], Bs[k], 1, 2, mode=mode)
                    assert int(ui[k]["score"]) == w.score and psa.unpack_ops(uo[k], int(ui[k]["aln_len"])) == w.ops
            c.close()
        except Exception as ex:           # reported by the main thread
            errors.append((t, repr(ex)))

    th = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors
