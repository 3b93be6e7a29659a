"""One banded pair over the whole GPU (psa_align_pair_banded, psa_align_long_banded_device): against the banded oracle,
against a one-pair psa_align_batch_banded (the one-warp path) record for record and op word for op word, against
psa_align_pair / psa_align_long_device when the band holds every cell, and at scale against the linear-space banded
oracle with fewer warps than row blocks."""
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
from tests.test_gpu_banded import in_band, rescore

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5A5A5A5
FIELDS = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j", "start_i", "start_j")
BANDS = [0, 1, 7, 31, 127, 128, 255, 256, 300, 1000]
SHAPES = [(300, 300), (3000, 3000), (900, 120), (120, 900), (513, 257), (1, 5000), (5000, 1), (37, 9000), (9000, 37),
          (3000, 20000)]
PENALTIES = [(1, 2), (0, 0), (0, 1), (2, 0), (3, 1), (5, 2)]


@pytest.fixture(scope="module")
def ctx():
    c = psa.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_one_cta():
    c = psa.Context(0)
    c.set_option("long_ctas_per_sm", 1)
    yield c
    c.close()


def words_for(m, n):
    return (m + n + 15) // 16 + 1


def expected_launches(m, n, band, tb):
    """The launch count include/psa.h documents for psa_align_long_banded_device."""
    if not tb:
        return 2
    bw = min(band, m + n)
    NB, S = -(-m // 128), -(-n // 256)
    tpr = min(S, (2 * bw + 128 * n // m + 2) // 256 + 2)
    rpw = min(NB, max(1, 2 ** 28 // (tpr * 16384)))
    return 2 + 2 * -(-NB // rpw)


def one_warp(ctx, a, b, band, mode, g=1, h=2, tb=True):
    """One-pair psa_align_batch_banded: (record, op words or None)."""
    ba, oa, la = psa.pack_pairs([a])
    bb, ob, lb = psa.pack_pairs([b])
    items, ops = ctx.align_batch_banded(ba, oa, la, bb, ob, lb, band, mode, g, h, traceback=tb)
    return items[0], (ops[0] if tb else None)


class Dev:
    """One pair resident on the device with a record and a sentinel-filled op buffer."""

    def __init__(self, a, b, stream):
        import torch
        with torch.cuda.stream(stream):
            self.a = torch.from_numpy(np.frombuffer(a, dtype=np.uint8).copy()).cuda()
            self.b = torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()
            self.words = words_for(len(a), len(b))
            self.item = torch.zeros(10, dtype=torch.int32, device="cuda")
            self.ops = torch.from_numpy(np.full(self.words, SENTINEL, dtype=np.uint32).view(np.int32)).cuda()
        stream.synchronize()
        self.m, self.n, self.stream = len(a), len(b), stream

    def run(self, ctx, band, mode, g=1, h=2, tb=True, banded=True):
        args = dict(mode=mode, g=g, h=h, traceback=tb, stream=self.stream.cuda_stream)
        if banded:
            ctx.align_long_banded_device(self.a.data_ptr(), self.b.data_ptr(), self.m, self.n, band, self.item.data_ptr(),
                                         self.ops.data_ptr() if tb else 0, self.words if tb else 0, **args)
        else:
            ctx.align_long_device(self.a.data_ptr(), self.b.data_ptr(), self.m, self.n, self.item.data_ptr(),
                                  self.ops.data_ptr() if tb else 0, self.words if tb else 0, **args)

    def result(self):
        return self.item.cpu().numpy().view(ITEM_DTYPE)[0].copy(), self.ops.cpu().numpy().view(np.uint32).copy()


def device(ctx, a, b, band, mode, g=1, h=2, tb=True):
    import torch
    st = torch.cuda.Stream()
    d = Dev(a, b, st)
    d.run(ctx, band, mode, g, h, tb)
    st.synchronize()
    return d.result()


def check_pair(ctx, a, b, band, mode, g=1, h=2, oracle=True, tag=""):
    """Both entries, with and without traceback, against the one-warp path (and the banded oracle)."""
    ref, ref_ops = one_warp(ctx, a, b, band, mode, g, h)
    L = int(ref["aln_len"])
    if oracle:
        w = bo.align_banded(a, b, band, g, h, mode)
        assert tuple(int(ref[f]) for f in FIELDS) == tuple(getattr(w, f) for f in FIELDS), (tag, ref, w)
        assert psa.unpack_ops(ref_ops, L) == w.ops, tag
    host = ctx.align_pair_banded(a, b, band, mode, g, h)
    assert tuple(getattr(host, f) for f in FIELDS) == tuple(int(ref[f]) for f in FIELDS), (tag, host, ref)
    assert host.ops == psa.unpack_ops(ref_ops, L), tag
    if L:
        assert (host.row_a, host.row_b) == psa.render_rows(a, b, host.ops, host.start_i, host.start_j), tag
    it, ops = device(ctx, a, b, band, mode, g, h)
    assert it.tobytes() == ref.tobytes(), (tag, it, ref)
    nw = (L + 15) // 16
    assert np.array_equal(ops[:nw], ref_ops[:nw]), tag
    assert (ops[nw:] == SENTINEL).all(), tag
    sref, _ = one_warp(ctx, a, b, band, mode, g, h, tb=False)
    shost = ctx.align_pair_banded(a, b, band, mode, g, h, traceback=False)
    assert tuple(getattr(shost, f) for f in FIELDS) == tuple(int(sref[f]) for f in FIELDS), (tag, shost, sref)
    sit, sops = device(ctx, a, b, band, mode, g, h, tb=False)
    assert sit.tobytes() == sref.tobytes(), (tag, sit, sref)
    assert (sops == SENTINEL).all()
    return ref


def pair_for(rng, m, n, related):
    a = random_dna(rng, m)
    return a, (mutated_copy(rng, a, n) if related else random_dna(rng, n))


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_shapes_and_bands_match_oracle_and_one_warp_path(ctx, mode):
    rng = np.random.default_rng(6100 + mode)
    for k, (m, n) in enumerate(SHAPES):
        a, b = pair_for(rng, m, n, k % 3 != 2)
        for band in BANDS + [max(m, n)]:
            if m * n > 10 ** 7 and band not in (31, 1000, max(m, n)):
                continue                  # the full-table oracle of the largest shape: three bands
            check_pair(ctx, a, b, band, mode, tag=f"{m}x{n} band {band}")


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_penalties_alphabets_and_ties(ctx, mode):
    rnd = random.Random(6200 + mode)
    rng = np.random.default_rng(6201 + mode)
    pairs = [pair_for(rng, 700, 650, True),
             (bytes(rnd.randrange(256) for _ in range(600)), bytes(rnd.randrange(256) for _ in range(540))),
             (bytes(rnd.choice(b"AB") for _ in range(800)), bytes(rnd.choice(b"AB") for _ in range(760)))]
    for motif in (b"AC", b"ACG", b"AACG"):
        pairs.append((motif * (700 // len(motif)), motif * (650 // len(motif)) + b"T"))
    for g, h in PENALTIES:
        for band in (0, 7, 128, 300):
            for a, b in pairs:
                check_pair(ctx, a, b, band, mode, g, h, tag=f"g{g} h{h} band {band} {len(a)}x{len(b)}")


def test_no_global_path(ctx):
    for a, b in ((b"A", b"ACGT" * 250), (b"AC", b"ACGT" * 250), (random_dna(np.random.default_rng(1), 40), b"ACGT" * 2000)):
        ref = check_pair(ctx, a, b, 10, psa.GLOBAL, tag=f"{len(a)}x{len(b)}")
        assert (int(ref["t1"]), int(ref["t2"]), int(ref["t3"]), int(ref["score"]), int(ref["end_state"]),
                int(ref["aln_len"])) == (NEG_INF, NEG_INF, NEG_INF, NEG_INF, 1, 0)


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_wide_band_equals_unbanded_entries(ctx, mode):
    import torch
    rng = np.random.default_rng(6300 + mode)
    for m, n in [(300, 300), (900, 120), (513, 257), (3000, 3000), (1500, 4000)]:
        a, b = pair_for(rng, m, n, True)
        for tb in (True, False):
            want = ctx.align_pair(a, b, mode, 1, 2, traceback=tb)
            got = ctx.align_pair_banded(a, b, max(m, n) + 3, mode, 1, 2, traceback=tb)
            for f in FIELDS + ("ops", "row_a", "row_b"):
                assert getattr(got, f) == getattr(want, f), (m, n, tb, f)
            st = torch.cuda.Stream()
            ref, banded = Dev(a, b, st), Dev(a, b, st)
            ref.run(ctx, 0, mode, tb=tb, banded=False)
            banded.run(ctx, max(m, n), mode, tb=tb)
            st.synchronize()
            (ri, ro), (bi, bo_) = ref.result(), banded.result()
            assert bi.tobytes() == ri.tobytes(), (m, n, tb)
            L = (int(ri["aln_len"]) + 15) // 16
            assert np.array_equal(bo_[:L], ro[:L]), (m, n, tb)


@pytest.mark.parametrize("band", [2000, 20000])
def test_wavefront_100kbp_against_linear_oracle(ctx, ctx_one_cta, band):
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    a, b = A[:100_000].tobytes(), B[:100_000].tobytes()
    for mode in (psa.GLOBAL, psa.LOCAL):
        want = bo.score_banded(a, b, band, 1, 2, mode)
        wt = (want.t1, want.t2, want.t3, want.score, want.end_state, want.end_i, want.end_j)
        for c in (ctx, ctx_one_cta):
            for tb in (False, True):
                r = c.align_pair_banded(a, b, band, mode, traceback=tb)
                assert (r.t1, r.t2, r.t3, r.score, r.end_state, r.end_i, r.end_j) == wt, (band, mode, tb, r)
                if tb:
                    assert rescore(a, b, r.ops, r.start_i, r.start_j, 1, 2, mode) == r.score, (band, mode)
                    assert in_band(a, b, r.ops, r.start_i, r.start_j, band), (band, mode)


@pytest.mark.parametrize("m,n", [(2_097_150, 257), (257, 2_097_150)])
def test_lengths_at_the_limit(ctx, m, n):
    rng = np.random.default_rng(6400)
    a, b = pair_for(rng, m, n, False)
    for mode in (psa.GLOBAL, psa.LOCAL):
        check_pair(ctx, a, b, 64, mode, oracle=False, tag=f"{m}x{n}")


def test_1Mbp_band_1000_traceback_equals_one_warp_path():
    import torch
    A, B = synth.mutated_pair(1_000_000, synth.SEED_C4)
    a, b = A.tobytes(), B.tobytes()
    torch.cuda.init()
    ref_ctx = psa.Context(0)
    ref, ref_ops = one_warp(ref_ctx, a, b, 1000, psa.GLOBAL)
    ref_ctx.close()
    free0, _ = torch.cuda.mem_get_info()
    c = psa.Context(0)
    got = c.align_pair_banded(a, b, 1000, psa.GLOBAL)
    free1, _ = torch.cuda.mem_get_info()
    c.close()
    used = free0 - free1
    print(f"1 Mbp banded pair traceback: context allocated {used / 2**30:.2f} GiB")
    assert used < 2 * 2**30, used
    assert tuple(getattr(got, f) for f in FIELDS) == tuple(int(ref[f]) for f in FIELDS)
    assert got.ops == psa.unpack_ops(ref_ops, int(ref["aln_len"]))
    assert rescore(a, b, got.ops, got.start_i, got.start_j, 1, 2, psa.GLOBAL) == got.score


def test_device_form_streams_sentinels_and_launch_count(ctx):
    import torch
    rng = np.random.default_rng(6500)
    cases = [pair_for(rng, 3000, 2500, True), pair_for(rng, 2000, 2000, False), pair_for(rng, 2_097_150, 257, False)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for (a, b), band, mode in zip(cases, (100, 31, 64), (psa.GLOBAL, psa.LOCAL, psa.GLOBAL)):
        for tb in (True, False):
            ref1, ref1_ops = one_warp(ctx, a, b, band, mode, tb=tb)
            ref2, ref2_ops = one_warp(ctx, b, a, band, mode, tb=tb)
            d1, d2 = Dev(a, b, s1), Dev(b, a, s2)
            n0 = ctx.launches
            d1.run(ctx, band, mode, tb=tb)
            assert ctx.launches - n0 == expected_launches(len(a), len(b), band, tb)
            d2.run(ctx, band, mode, tb=tb)             # right after, on another stream of the same context
            s1.synchronize()                           # the first call is complete once its own stream is
            for d, ref, ref_ops in ((d1, ref1, ref1_ops), (d2, ref2, ref2_ops)):
                if d is d2:
                    s2.synchronize()
                it, ops = d.result()
                assert it.tobytes() == ref.tobytes(), (len(a), band, tb)
                L = (int(it["aln_len"]) + 15) // 16 if tb else 0
                if tb:
                    assert np.array_equal(ops[:L], ref_ops[:L])
                assert (ops[L:] == SENTINEL).all()


def test_errors(ctx):
    import torch
    a, b = b"ACGT" * 100, b"ACGA" * 100
    for kw, code in ((dict(band=-1), -1), (dict(band=5, flags=psa.WANT_SCORE | psa.OPS_COMPACT), -1), (dict(band=5, mode=7), -1),
                     (dict(band=5, g=-1), -1)):
        with pytest.raises(PsaError) as e:
            ctx.align_pair_banded(a, b, **kw)
        assert e.value.code == code, kw
    with pytest.raises(PsaError) as e:
        ctx.align_pair_banded(b"A" * (2 ** 21 - 1), b"ACGT", 10, traceback=False)
    assert e.value.code == -2
    # m == 0 or n == 0: psa_align_pair's record
    for x, y in ((b"", b"ACGT"), (b"ACG", b"")):
        for mode in (psa.GLOBAL, psa.LOCAL):
            got, want = ctx.align_pair_banded(x, y, 3, mode), ctx.align_pair(x, y, mode)
            assert all(getattr(got, f) == getattr(want, f) for f in FIELDS + ("ops", "row_a", "row_b")), (x, y, mode)
    st = torch.cuda.Stream()
    d = Dev(a, b, st)
    with pytest.raises(PsaError) as e:
        ctx.align_long_banded_device(d.a.data_ptr(), d.b.data_ptr(), 400, 400, 5, d.item.data_ptr(), d.ops.data_ptr(), 49,
                                     traceback=True, stream=st.cuda_stream)
    assert e.value.code == -5
    with pytest.raises(PsaError) as e:
        ctx.align_long_banded_device(d.a.data_ptr(), d.b.data_ptr(), 400, 400, 5, d.item.data_ptr(), 0, 0, traceback=True)
    assert e.value.code == -5
    for m, n, band, flags in ((0, 400, 5, psa.WANT_SCORE), (400, 400, -2, psa.WANT_SCORE), (400, 400, 5, 8)):
        with pytest.raises(PsaError) as e:
            ctx.align_long_banded_device(d.a.data_ptr(), d.b.data_ptr(), m, n, band, d.item.data_ptr(), flags=flags)
        assert e.value.code == -1, (m, n, band, flags)
    with pytest.raises(PsaError) as e:
        ctx.align_long_banded_device(d.a.data_ptr(), d.b.data_ptr(), 2 ** 21 - 1, 400, 5, d.item.data_ptr())
    assert e.value.code == -2


def test_threads_mix_pair_batch_and_unbanded():
    errors = []

    def work(t):
        try:
            c = psa.Context(0)
            rng = np.random.default_rng(6600 + t)
            mode = psa.LOCAL if t % 2 else psa.GLOBAL
            for band in (7, 64, 300):
                a, b = pair_for(rng, int(rng.integers(300, 1500)), int(rng.integers(300, 1500)), True)
                w = bo.align_banded(a, b, band, 1, 2, mode)
                r = c.align_pair_banded(a, b, band, mode)
                assert (r.score, r.end_i, r.end_j, r.ops) == (w.score, w.end_i, w.end_j, w.ops), (t, band)
                items, ops = one_warp(c, a, b, band, mode)
                assert psa.unpack_ops(ops, int(items["aln_len"])) == w.ops, (t, band)
                u = c.align_pair(a, b, mode)
                wu = po.align(a, b, 1, 2, mode=mode)
                assert (u.score, u.ops) == (wu.score, wu.ops), (t, band)
            c.close()
        except Exception as ex:           # reported by the main thread
            errors.append((t, repr(ex)))

    th = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors
