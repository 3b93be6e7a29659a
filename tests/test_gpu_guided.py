"""Banded alignment along an anchor chain (psa_align_batch_guided[_device], psa_align_pair_guided): the empty chain
against the diagonal band entries, wide bands against psa_align_batch, random chains against the per-row oracle on all
three entries, structural-variant pairs that only a chain reaches at a narrow band, the device form's rejected record,
chunking, the whole-GPU pair path against the one-warp batch, launch counts and host threads."""
import random
import threading

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200 import synth
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE, NEG_INF, PsaError
from oracle import pyoracle as po
from tests import banded_oracle as bo
from tests import guided_oracle as go
from tests.helpers import mutated_copy, random_dna
from tests.test_gpu_banded import FIELDS, SENTINEL, _narrow_cases, rescore
from tests.test_guided_cpu import random_chain, rowblock_tiles

pytestmark = pytest.mark.gpu

BANDS = [0, 1, 7, 127, 128, 300]


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


def _host(ctx, As, Bs, chains, band, mode, g=1, h=2, tb=True):
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    return ctx.align_batch_guided(ba, oa, la, bb, ob, lb, chains, band, mode, g, h, traceback=tb)


def _banded(ctx, As, Bs, band, mode, tb=True):
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    return ctx.align_batch_banded(ba, oa, la, bb, ob, lb, band, mode, traceback=tb)


def _device(ctx, As, Bs, chains, band, mode, g=1, h=2, tb=True, raw=None):
    """The device entry on torch tensors and a side stream; op words start as a sentinel.  raw: (anchors, off, cnt)
    arrays passed as they are (invalid chains included)."""
    import torch
    dev = torch.device("cuda", 0)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    anc, off, cnt = raw if raw is not None else psa.pack_anchors(chains)
    n, stride = len(As), _stride(As, Bs)
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        pad = np.zeros(1, dtype=np.uint8)
        t = [torch.from_numpy(x).to(dev) for x in (np.concatenate([ba, pad]), oa, la, np.concatenate([bb, pad]), ob, lb,
                                                   np.concatenate([anc.reshape(-1), np.zeros(2, np.int32)]), off, cnt)]
        items = torch.zeros(n * 10, dtype=torch.int32, device=dev)
        ops = torch.from_numpy(np.full(n * stride, SENTINEL, dtype=np.uint32).view(np.int32)).to(dev)
        st.synchronize()
        ctx.align_batch_guided_device(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                                      t[5].data_ptr(), n, int(la.max()), int(lb.max()), t[6].data_ptr(), t[7].data_ptr(),
                                      t[8].data_ptr(), band, items.data_ptr(), ops.data_ptr() if tb else 0, stride if tb else 0,
                                      mode, g, h, tb, st.cuda_stream)
        st.synchronize()
    return items.cpu().numpy().view(ITEM_DTYPE).copy(), ops.cpu().numpy().view(np.uint32).reshape(n, stride).copy()


def _pair_items(ctx, As, Bs, chains, band, mode, tb=True):
    """psa_align_pair_guided on every pair, as batch records and op words."""
    items = np.zeros(len(As), dtype=ITEM_DTYPE)
    ops = np.zeros((len(As), _stride(As, Bs)), dtype=np.uint32)
    for k, (a, b) in enumerate(zip(As, Bs)):
        r = ctx.align_pair_guided(a, b, chains[k], band, mode, traceback=tb)
        items[k] = (r.t1, r.t2, r.t3, r.score, r.end_state, r.end_i, r.end_j, r.start_i, r.start_j, len(r.ops))
        w = np.zeros(ops.shape[1], np.uint32)
        for q, o in enumerate(reversed(r.ops)):          # forward bytes -> traceback-order words
            w[q >> 4] |= np.uint32(o) << np.uint32(2 * (q & 15))
        ops[k] = w
    return items, ops


def in_rows(ops, start_i, start_j, lo, hi):
    i, j = start_i, start_j
    for k, t in enumerate(ops):
        if k:
            i += t != 2
            j += t != 3
        if not lo[i] <= j <= hi[i]:
            return False
    return True


def check_rows(As, Bs, chains, items, ops, band, mode, tb=True, tag=""):
    for k, (a, b) in enumerate(zip(As, Bs)):
        lo, hi = go.guide_rows(len(a), len(b), chains[k], band)
        w = go.align_rows(a, b, lo, hi, 1, 2, mode)
        it = items[k]
        assert tuple(int(it[f]) for f in FIELDS) == tuple(getattr(w, f) for f in FIELDS), (tag, k, len(a), len(b), band, it, w)
        if not tb:
            assert int(it["aln_len"]) == 0
            continue
        assert (int(it["start_i"]), int(it["start_j"]), int(it["aln_len"])) == (w.start_i, w.start_j, len(w.ops)), (tag, k)
        got = psa.unpack_ops(ops[k], int(it["aln_len"]))
        assert got == w.ops, (tag, k, band)
        if w.score != po.NEG and len(a) and len(b):
            assert in_rows(got, w.start_i, w.start_j, lo, hi), (tag, k)
            assert rescore(a, b, got, w.start_i, w.start_j, 1, 2, mode) == w.score, (tag, k)


def _same(x, y):
    (ia, oa), (ib, ob) = x, y
    assert ia.tobytes() == ib.tobytes()
    for k in range(len(ia)):
        L = (int(ia[k]["aln_len"]) + 15) // 16
        assert np.array_equal(oa[k, :L], ob[k, :L]), k


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_empty_chain_equals_diagonal_band(ctx, mode):
    rng = np.random.default_rng(9000 + mode)
    As, Bs = _narrow_cases(rng, random.Random(9001 + mode))
    chains = [[]] * len(As)
    for band in BANDS:
        for tb in (True, False):
            want = _banded(ctx, As, Bs, band, mode, tb)
            got = _host(ctx, As, Bs, chains, band, mode, tb=tb)
            assert got[0].tobytes() == want[0].tobytes(), (band, tb)
            if tb:
                _same(got, want)
            d = _device(ctx, As, Bs, chains, band, mode, tb=tb)
            assert d[0].tobytes() == want[0].tobytes(), (band, tb)
        for a, b in zip(As, Bs):
            if not (a and b):
                continue
            for tb in (True, False):
                n0 = ctx.launches
                r1 = ctx.align_pair_banded(a, b, band, mode, traceback=tb)
                n1 = ctx.launches
                r2 = ctx.align_pair_guided(a, b, [], band, mode, traceback=tb)
                assert ctx.launches - n1 == n1 - n0
                assert [getattr(r1, f) for f in r1.__slots__] == [getattr(r2, f) for f in r2.__slots__]


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_wide_band_equals_align_batch(ctx, mode):
    rng = np.random.default_rng(9100 + mode)
    rnd = random.Random(9101 + mode)
    As = [random_dna(rng, int(rng.integers(257, 1500))) for _ in range(10)]
    Bs = [mutated_copy(rng, a, int(rng.integers(257, 1500))) if k % 2 else random_dna(rng, int(rng.integers(257, 1500)))
          for k, a in enumerate(As)]
    chains = [random_chain(rnd, len(a), len(b), rnd.choice([0, 1, 4, 20])) for a, b in zip(As, Bs)]
    band = max(map(len, As + Bs))
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    want = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=True)
    _same(_host(ctx, As, Bs, chains, band, mode), want)
    _same(_device(ctx, As, Bs, chains, band, mode), want)
    _same(_pair_items(ctx, As[:4], Bs[:4], chains[:4], band, mode), (want[0][:4], want[1][:4, :_stride(As[:4], Bs[:4])]))
    ws, _ = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=False)
    assert _host(ctx, As, Bs, chains, band, mode, tb=False)[0].tobytes() == ws.tobytes()


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_random_chains_match_row_oracle(ctx, mode):
    rng = np.random.default_rng(9200 + mode)
    rnd = random.Random(9201 + mode)
    As, Bs = _narrow_cases(rng, rnd)
    for band in (0, 1, 7, 64, 300):
        chains = [random_chain(rnd, len(a), len(b), rnd.choice([0, 1, 2, 5, 16])) for a, b in zip(As, Bs)]
        items, ops = _device(ctx, As, Bs, chains, band, mode)
        check_rows(As, Bs, chains, items, ops, band, mode, tag=f"device {band}")
        for k, it in enumerate(items):
            if int(it["aln_len"]) == 0:
                assert (ops[k] == SENTINEL).all(), (band, k)
        h = _host(ctx, As, Bs, chains, band, mode)
        assert h[0].tobytes() == items.tobytes(), band
        s = _host(ctx, As, Bs, chains, band, mode, tb=False)[0]
        check_rows(As, Bs, chains, s, None, band, mode, tb=False, tag=f"score {band}")
        keep = [k for k in range(len(As)) if len(As[k]) and len(Bs[k])][:6]
        sub = [As[k] for k in keep], [Bs[k] for k in keep], [chains[k] for k in keep]
        pi, po_ = _pair_items(ctx, *sub, band, mode)
        check_rows(*sub, pi, po_, band, mode, tag=f"pair {band}")


def sv_pair(seed):
    """A 5 kbp pair with one 500 - 2000 bp insertion in A (even seeds) or in B (odd seeds), 3 % substitutions, and the
    chain at the true breakpoints: a vertical or a horizontal run."""
    rng = np.random.default_rng(seed)
    x = random_dna(rng, 5000)
    y = mutated_copy(rng, x, 5000, sub=0.03, ins=0.0, dele=0.0)
    L, p = int(rng.integers(500, 2001)), int(rng.integers(1000, 4000))
    ins = random_dna(rng, L)
    if seed % 2 == 0:
        return x[:p] + ins + x[p:], y, [[p, p], [p + L, p]]
    return x, y[:p] + ins + y[p:], [[p, p], [p, p + L]]


def test_structural_variants_reach_the_unbanded_optimum(ctx):
    """At band 64 the chain finds the global optimum of psa_align_batch; the diagonal band of the same width does not."""
    As, Bs, chains = zip(*[sv_pair(s) for s in range(9100, 9110)])
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    full, full_ops = ctx.align_batch(ba, oa, la, bb, ob, lb, psa.GLOBAL, 1, 2, traceback=True)
    items, ops = _host(ctx, As, Bs, chains, 64, psa.GLOBAL)
    plain, _ = _banded(ctx, As, Bs, 64, psa.GLOBAL, tb=False)
    for k, (a, b) in enumerate(zip(As, Bs)):
        lin = po.score_linear(a, b, 1, 2, mode=po.GLOBAL)
        it = items[k]
        assert tuple(int(it[f]) for f in FIELDS) == tuple(int(full[k][f]) for f in FIELDS) == \
               (lin.t1, lin.t2, lin.t3, lin.score, lin.end_state, lin.end_i, lin.end_j), k
        got = psa.unpack_ops(ops[k], int(it["aln_len"]))
        assert rescore(a, b, got, int(it["start_i"]), int(it["start_j"]), 1, 2, psa.GLOBAL) == lin.score
        lo, hi = go.guide_rows(len(a), len(b), chains[k], 64)
        assert in_rows(got, int(it["start_i"]), int(it["start_j"]), lo, hi)
        assert int(plain[k]["score"]) < lin.score, k


def test_device_rejects_invalid_chains(ctx):
    rng = np.random.default_rng(9300)
    rnd = random.Random(9301)
    As = [random_dna(rng, int(rng.integers(300, 900))) for _ in range(10)]
    Bs = [mutated_copy(rng, a, int(rng.integers(300, 900))) for a in As]
    chains = [random_chain(rnd, len(a), len(b), rnd.choice([0, 3, 8])) for a, b in zip(As, Bs)]
    bad = {1: [[5, 5], [4, 9]], 3: [[len(As[3]) + 1, 2]], 4: [[3, -1]], 6: [[10, 10], [20, 9]], 8: None}
    for mode in (psa.GLOBAL, psa.LOCAL):
        for tb in (True, False):
            mixed = [np.array(bad[k], np.int32).reshape(-1, 2) if k in bad and bad[k] is not None else chains[k]
                     for k in range(len(As))]
            anc, off, cnt = psa.pack_anchors(mixed)
            cnt = cnt.copy()
            cnt[8] = -1                                  # a negative anchor count
            items, ops = _device(ctx, As, Bs, None, 40, mode, tb=tb, raw=(anc, off, cnt))
            good = [k for k in range(len(As)) if k not in bad]
            ref = _device(ctx, [As[k] for k in good], [Bs[k] for k in good], [chains[k] for k in good], 40, mode, tb=tb)
            for k in bad:
                it = items[k]
                assert tuple(int(it[f]) for f in ITEM_DTYPE.names) == (NEG_INF,) * 4 + (0,) * 6, (k, it)
                assert (ops[k] == SENTINEL).all(), k
            for q, k in enumerate(good):
                assert items[k].tobytes() == ref[0][q].tobytes(), k
                if tb:
                    L = (int(items[k]["aln_len"]) + 15) // 16
                    assert np.array_equal(ops[k, :L], ref[1][q, :L]), k
    # the host forms refuse the same chains, naming the pair and the anchor
    for k in bad:
        if bad[k] is None:
            continue
        mixed = list(chains)
        mixed[k] = bad[k]
        with pytest.raises(PsaError) as e:
            _host(ctx, As, Bs, mixed, 40, psa.GLOBAL)
        assert e.value.code == -1 and f"pair {k}" in str(e.value), str(e.value)
        with pytest.raises(PsaError) as e:
            ctx.align_pair_guided(As[k], Bs[k], bad[k], 40)
        assert e.value.code == -1 and "anchor" in str(e.value)


def test_argument_errors(ctx):
    As, Bs = [b"ACGT" * 100], [b"ACGA" * 100]
    for call in (lambda: _host(ctx, As, Bs, [[]], -1, psa.GLOBAL), lambda: ctx.align_pair_guided(As[0], Bs[0], [], -1),
                 lambda: _device(ctx, As, Bs, [[]], -3, psa.LOCAL),
                 lambda: ctx.align_pair_guided(As[0], Bs[0], [], 10, flags=psa.WANT_SCORE | psa.OPS_COMPACT, traceback=False)):
        with pytest.raises(PsaError) as e:
            call()
        assert e.value.code == -1
    big = b"A" * (2 ** 21 - 1)
    with pytest.raises(PsaError) as e:
        _host(ctx, [big], [b"ACGT"], [[]], 10, psa.GLOBAL, tb=False)
    assert e.value.code == -2
    with pytest.raises(PsaError) as e:
        ctx.align_pair_guided(big, b"ACGT", [], 10)
    assert e.value.code == -2
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    with pytest.raises(PsaError) as e:
        ctx.align_batch_guided(ba, oa, la, bb, ob, lb, [[]], 10, ops=np.zeros((1, 49), dtype=np.uint32))
    assert e.value.code == -5
    # an anchor range past the end of the anchor array
    anc, off, cnt = psa.pack_anchors([[[1, 1], [2, 2]]])
    out = np.zeros(1, ITEM_DTYPE)
    with pytest.raises(PsaError) as e:
        ctx._check(ctx._lib.psa_align_batch_guided(ctx._h, ba.ctypes.data, oa.ctypes.data, la.ctypes.data, bb.ctypes.data,
                                                   ob.ctypes.data, lb.ctypes.data, 1, ba.size, bb.size, anc.ctypes.data,
                                                   off.ctypes.data, cnt.ctypes.data, 1, 0, 1, 2, 10, 1,
                                                   out.ctypes.data, None, 0))
    assert e.value.code == -1 and "pair 0" in str(e.value)
    # empty sides: psa_align_batch's record
    r = ctx.align_pair_guided(b"", b"ACG", [], 3)
    w = ctx.align_pair(b"", b"ACG")
    assert (r.t1, r.t2, r.t3, r.score, r.ops) == (w.t1, w.t2, w.t3, w.score, w.ops)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_chunked_equals_one_chunk(ctx, ctx_chunked, mode):
    rng = np.random.default_rng(9400 + mode)
    rnd = random.Random(9401 + mode)
    As = [random_dna(rng, int(rng.integers(300, 1500))) for _ in range(10)]
    Bs = [mutated_copy(rng, a, int(rng.integers(300, 1500))) for a in As]
    chains = [random_chain(rnd, len(a), len(b), 6) for a, b in zip(As, Bs)]
    for band in (31, 256):
        one = _device(ctx, As, Bs, chains, band, mode)
        many = _device(ctx_chunked, As, Bs, chains, band, mode)
        assert one[0].tobytes() == many[0].tobytes() and np.array_equal(one[1], many[1]), band
        check_rows(As, Bs, chains, one[0], one[1], band, mode)


def documented_launches(m, n, chain, band, tb):
    """include/psa.h's launch count of psa_align_pair_guided."""
    if not tb:
        return 2
    NB = (m + 127) // 128
    bw = min(band, m + n)
    if len(chain) == 0:
        tpr = min((n + 255) // 256, (2 * bw + 128 * n // m + 2) // 256 + 2)
    else:
        lo, hi = go.guide_rows(m, n, chain, bw)
        tpr = max(rowblock_tiles(lo, hi, m))
    rpw = min(NB, max(1, (1 << 28) // (tpr * 16384)))
    return 2 + 2 * ((NB + rpw - 1) // rpw)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_whole_gpu_pair_equals_one_warp_batch_at_100kbp(ctx, mode):
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    a, b = A[:100_000].tobytes(), B[:100_000].tobytes()
    rnd = random.Random(9500 + mode)
    chain = [[0, 0]]
    for i in range(20_000, 100_000, 20_000):        # a multi-segment chain near the diagonal, with small detours
        d = rnd.randint(-300, 300)
        chain.append([i, max(chain[-1][1], i + d)])
    chain = np.array(chain, np.int32)
    lo, hi = go.guide_rows(len(a), len(b), chain, 400)
    want = go.score_rows(a, b, lo, hi, 1, 2, mode)
    for tb in (True, False):
        n0 = ctx.launches
        r = ctx.align_pair_guided(a, b, chain, 400, mode, traceback=tb)
        assert ctx.launches - n0 == documented_launches(len(a), len(b), chain, 400, tb)
        assert (r.t1, r.t2, r.t3, r.score, r.end_state, r.end_i, r.end_j) == \
               (want.t1, want.t2, want.t3, want.score, want.end_state, want.end_i, want.end_j), tb
        bi, bops = _host(ctx, [a], [b], [chain], 400, mode, tb=tb)
        assert (int(bi[0]["score"]), int(bi[0]["end_i"]), int(bi[0]["end_j"])) == (r.score, r.end_i, r.end_j)
        if tb:
            assert (int(bi[0]["start_i"]), int(bi[0]["start_j"]), int(bi[0]["end_state"])) == (r.start_i, r.start_j, r.end_state)
            assert psa.unpack_ops(bops[0], int(bi[0]["aln_len"])) == r.ops


def test_1Mbp_two_indels_traceback_in_one_call_on_the_pair_path():
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    rng = np.random.default_rng(9600)
    i1, i2 = random_dna(rng, 10_000), random_dna(rng, 10_000)
    a = A[:300_000].tobytes() + i1 + A[300_000:].tobytes()
    b = B[:700_000].tobytes() + i2 + B[700_000:].tobytes()
    # breakpoints: A's insertion is a vertical run at row 300 000, B's a horizontal run at row 710 000 (A's coordinates
    # are 10 kbp ahead after the first insertion)
    chain = np.array([[300_000, 300_000], [310_000, 300_000], [710_000, 700_000], [710_000, 710_000]], np.int32)
    c = psa.Context(0)
    n0 = c.launches
    r = c.align_pair_guided(a, b, chain, 100, psa.GLOBAL)
    assert c.launches - n0 == documented_launches(len(a), len(b), chain, 100, True)
    c.close()
    assert r.score > NEG_INF and len(r.ops) >= len(a)
    assert rescore(a, b, r.ops, r.start_i, r.start_j, 1, 2, psa.GLOBAL) == r.score
    lo, hi = go.guide_rows(len(a), len(b), chain, 100)
    assert in_rows(r.ops, r.start_i, r.start_j, lo, hi)


def test_threads_mix_guided_banded_and_unbanded():
    errors = []

    def work(t):
        try:
            c = psa.Context(0)
            rng = np.random.default_rng(9700 + t)
            rnd = random.Random(9700 + t)
            mode = psa.LOCAL if t % 2 else psa.GLOBAL
            for band in (7, 64, 300):
                As = [random_dna(rng, int(rng.integers(200, 700))) for _ in range(5)]
                Bs = [mutated_copy(rng, a, int(rng.integers(200, 700))) for a in As]
                chains = [random_chain(rnd, len(a), len(b), 4) for a, b in zip(As, Bs)]
                items, ops = _host(c, As, Bs, chains, band, mode)
                check_rows(As, Bs, chains, items, ops, band, mode)
                bi, _ = _banded(c, As, Bs, band, mode, tb=False)
                ui, _ = c.align_batch(*psa.pack_pairs(As), *psa.pack_pairs(Bs), mode, 1, 2, traceback=False)
                for k in range(len(As)):
                    assert int(bi[k]["score"]) == bo.score_banded(As[k], Bs[k], band, 1, 2, mode).score
                    assert int(ui[k]["score"]) == po.score_linear(As[k], Bs[k], 1, 2, mode=mode).score
            c.close()
        except Exception as ex:           # reported by the main thread
            errors.append((t, repr(ex)))

    # the CPU oracles build their libraries on first use; build them here, not concurrently in the threads
    bo.lib(), go.lib(), po.lib()
    th = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors
