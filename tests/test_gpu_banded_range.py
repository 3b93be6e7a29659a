"""The four banded entries (psa_align_batch_banded[_device], psa_align_pair_banded, psa_align_long_banded_device) at the
edge of the scoring range, against the exact banded reference (tests/banded_exact.py).

A band can force a gap opening on every row, so global calls with band < max(m, n) are held to check_banded_scoring's
bound g(m+n+2) + h(min(m, n) + 3) + m + n < 2^28 rather than the full matrix's three openings.  At the largest penalties
that bound admits, every entry equals the exact reference: record fields, op words (the same words on every entry, none
written past the alignment), a path that re-scores exactly to the score and stays in the band.  One unit more is
PSA_ERR_RANGE.  Penalties the old rule admitted never give a wrong record.  Local mode and bands that hold every cell keep
the unbanded limit.  Pairs without a path in the band still give the no-path record at the limit.  Local score-only
fills with 16 columns per lane find a best cell next to the padding columns at the largest h."""
import functools

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200.capi import NEG_INF, PsaError
from oracle import pyoracle as po
from tests import banded_exact as bx
from tests.helpers import random_dna
from tests.test_banded_range_cpu import EDGE_SHAPES, OLD_RULE_CASES, edge_pair, edge_penalties
from tests.test_gpu_banded import _device as batch_device
from tests.test_gpu_banded import in_band, rescore
from tests.test_gpu_banded_pair import device as pair_device

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5A5A5A5
ERR_RANGE = -2
MODES = [psa.GLOBAL, psa.LOCAL]


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


@functools.lru_cache(maxsize=None)
def exact(a, b, band, g, h, mode):
    return bx.align_banded(a, b, band, g, h, mode)


# ---- the four entries on one pair: (record as 10 ints in psa_batch_item order, ops, op words or None) --------------

def _record(item, words, tb):
    """(the 10 fields, forward ops, the op words that carry them, whether every word past those is untouched)"""
    L = int(item["aln_len"])
    nw = (L + 15) // 16
    return tuple(item.tolist()), psa.unpack_ops(words, L) if tb else b"", words[:nw], bool((words[nw:] == SENTINEL).all())


def run_batch(ctx, a, b, band, mode, g, h, tb):
    ba, oa, la = psa.pack_pairs([a])
    bb, ob, lb = psa.pack_pairs([b])
    items, ops = ctx.align_batch_banded(ba, oa, la, bb, ob, lb, band, mode, g, h, traceback=tb)
    rec, got, words, _ = _record(items[0], ops[0] if tb else np.zeros(0, np.uint32), tb)
    return rec, got, words, True            # the host form copies the whole device stride back: no sentinel to check


def run_batch_device(ctx, a, b, band, mode, g, h, tb):
    items, ops = batch_device(ctx, [a], [b], band, mode, g, h, tb)
    return _record(items[0], ops[0], tb)


def run_pair(ctx, a, b, band, mode, g, h, tb):
    r = ctx.align_pair_banded(a, b, band, mode, g, h, traceback=tb)
    if r.ops:
        assert (r.row_a, r.row_b) == bx.render_rows(a, b, r.ops, r.start_i, r.start_j)
    rec = (r.t1, r.t2, r.t3, r.score, r.end_state, r.end_i, r.end_j, r.start_i, r.start_j, len(r.ops))
    return rec, r.ops, None, True


def run_long_device(ctx, a, b, band, mode, g, h, tb):
    item, ops = pair_device(ctx, a, b, band, mode, g, h, tb)
    return _record(item, ops, tb)


ENTRIES = {"batch": run_batch, "batch_device": run_batch_device, "pair": run_pair, "long_device": run_long_device}


def check(ctx, a, b, band, mode, g, h, entries=ENTRIES, tag=""):
    """Every entry, with and without traceback, against the exact reference."""
    w = exact(a, b, band, g, h, mode)
    for tb in (True, False):
        want = (w.t1, w.t2, w.t3, w.score, w.end_state, w.end_i, w.end_j) + \
               ((w.start_i, w.start_j, len(w.ops)) if tb else (0, 0, 0))
        words = []
        for name in entries:
            rec, ops, wd, untouched = ENTRIES[name](ctx, a, b, band, mode, g, h, tb)
            t = (tag, name, tb, g, h)
            assert rec == want, (t, rec, want)
            assert ops == (w.ops if tb else b""), t
            assert untouched, t                      # no op word written past the alignment
            if wd is not None:
                words.append(wd)
            if tb and ops:
                assert rescore(a, b, ops, rec[7], rec[8], g, h, mode) == w.score, t
                assert in_band(a, b, ops, rec[7], rec[8], band), t
        assert all(np.array_equal(x, words[0]) for x in words), (tag, tb)
    return w


def expect_range_error(ctx, a, b, band, mode, g, h, entries=ENTRIES, tag=""):
    for name in entries:
        for tb in (True, False):
            with pytest.raises(PsaError) as e:
                ENTRIES[name](ctx, a, b, band, mode, g, h, tb)
            assert e.value.code == ERR_RANGE, (tag, name, tb, g, h)
            assert "int32" in str(e.value)


# ---- (a) the largest admitted penalties ------------------------------------------------------------------------

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape", EDGE_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}_band{s[2]}")
def test_largest_admitted_penalties(ctx, shape, mode):
    """All four entries at the largest h (g = 0, 3) and g (h = 0, 2) check_banded_scoring admits; in global mode one
    unit more is PSA_ERR_RANGE on every entry, and the same context answers exactly right after."""
    m, n, band, related = shape
    a, b = edge_pair(m, n, related, m + band)
    lowest = 0
    for (g, h), over in edge_penalties(m, n):
        if mode == psa.GLOBAL:
            expect_range_error(ctx, a, b, band, mode, *over, tag=shape)
        w = check(ctx, a, b, band, mode, g, h, tag=shape)
        lowest = min([lowest] + [v for v in (w.t1, w.t2, w.t3) if v != NEG_INF])
    if mode == psa.GLOBAL and band == 1 and 3 * min(m, n) == max(m, n):
        assert lowest < -(1 << 27)             # the corners reach the edge the rule guards


def test_largest_admitted_penalties_20k_x_60k(ctx, ctx_one_cta):
    """One 20 000 x 60 000 pair at band 1 (an opening on each of 20 000 rows) through the one-pair entries, on the
    default context and with one CTA per SM."""
    m, n = 20_000, 60_000
    a, b = edge_pair(m, n, False, 20_001)
    for mode in MODES:
        for (g, h), over in edge_penalties(m, n):
            for c in (ctx, ctx_one_cta):
                if mode == psa.GLOBAL:
                    expect_range_error(c, a, b, 1, mode, *over, entries=("pair", "long_device"))
                w = check(c, a, b, 1, mode, g, h, entries=("pair", "long_device"), tag=(mode, g, h))
            if mode == psa.GLOBAL and g in (0, 3):
                assert w.score < -(1 << 27)


def test_batch_rule_takes_the_largest_lengths(ctx):
    """A batch is held to the bound of (max m, max n, min(max m, max n)): a 300 x 900 and a 900 x 300 pair together
    admit h up to the 900 x 900 limit, one more is refused although each pair alone would be admitted."""
    a1, b1 = edge_pair(300, 900, False, 301)
    a2, b2 = edge_pair(900, 300, False, 901)
    h = bx.largest_h(900, 900, 0)
    assert bx.span_banded(0, h + 1, 300, 900) < bx.SPAN_LIMIT
    for tb in (True, False):
        ba, oa, la = psa.pack_pairs([a1, a2])
        bb, ob, lb = psa.pack_pairs([b1, b2])
        items, ops = ctx.align_batch_banded(ba, oa, la, bb, ob, lb, 1, psa.GLOBAL, 0, h, traceback=tb)
        ditems, dops = batch_device(ctx, [a1, a2], [b1, b2], 1, psa.GLOBAL, 0, h, tb)
        assert items.tobytes() == ditems.tobytes()
        for k, (a, b) in enumerate(((a1, b1), (a2, b2))):
            w = exact(a, b, 1, 0, h, psa.GLOBAL)
            assert int(items[k]["score"]) == w.score
            if tb:
                assert psa.unpack_ops(ops[k], int(items[k]["aln_len"])) == w.ops
                assert psa.unpack_ops(dops[k], int(items[k]["aln_len"])) == w.ops
        assert exact(a1, b1, 1, 0, h, psa.GLOBAL).score < -(1 << 26)        # n = 3m: an opening on each of the 300 rows
        for call in (lambda: ctx.align_batch_banded(ba, oa, la, bb, ob, lb, 1, psa.GLOBAL, 0, h + 1, traceback=tb),
                     lambda: batch_device(ctx, [a1, a2], [b1, b2], 1, psa.GLOBAL, 0, h + 1, tb)):
            with pytest.raises(PsaError) as e:
                call()
            assert e.value.code == ERR_RANGE


# ---- (b) penalties the old rule admitted: the exact record or PSA_ERR_RANGE, never a wrong record ----------------

@pytest.mark.parametrize("case", OLD_RULE_CASES, ids=["2000x4000_band1", "600x1200_band1", "300x2400_band40"])
def test_no_wrong_records_where_the_old_rule_admitted(ctx, case):
    """Every entry returns the exact record or PSA_ERR_RANGE.  Under the three-openings rule all three were admitted and
    came back as the no-path record (PSA_NEG_INF corners, aln_len 0)."""
    m, n, band, g, h = case
    a, b = edge_pair(m, n, False, m + band)
    assert bx.span(g, h, m, n) < bx.SPAN_LIMIT
    w = exact(a, b, band, g, h, psa.GLOBAL)
    for name in ENTRIES:
        for tb in (True, False):
            try:
                rec, ops, _, _ = ENTRIES[name](ctx, a, b, band, psa.GLOBAL, g, h, tb)
            except PsaError as e:
                assert e.code == ERR_RANGE, (name, tb)
                continue
            assert rec[:7] == (w.t1, w.t2, w.t3, w.score, w.end_state, w.end_i, w.end_j), (name, tb, rec, w.score)
            if tb:
                assert ops == w.ops, (name, tb)
    # the context still answers exactly after the refusals
    a, b = edge_pair(300, 900, False, 301)
    check(ctx, a, b, 1, psa.GLOBAL, 1, 2)


# ---- (c) local mode keeps the unbanded limit -----------------------------------------------------------------

@pytest.mark.parametrize("shape", EDGE_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}_band{s[2]}")
def test_local_mode_at_the_unbanded_limit(ctx, shape):
    m, n, band, related = shape
    a, b = edge_pair(m, n, related, m + band)
    for g, h in ((0, bx.largest_h(m, n, 0, bx.span)), (bx.largest_g(m, n, 0, bx.span), 0)):
        assert bx.span_banded(g, h, m, n) >= bx.SPAN_LIMIT or h == 0
        check(ctx, a, b, band, psa.LOCAL, g, h, tag=shape)


def test_local_best_next_to_padding_columns(ctx):
    """Local score only at the largest h check_scoring admits, on the kernels with 16 columns per lane in the TF form
    (banded batches, the unbanded long batch, single-pair geometries 2 and 3).  Each best alignment ends in the lane that
    holds column n next to padding columns (n % 16 != 0).  A padding column's key used to wrap to a large positive value
    once g + h > 2^26 and hide that lane's best: this 900 x 300 case reported 95 where the oracle gives 98."""
    rng = np.random.default_rng(7300)
    As, Bs = [], []
    for n in range(300, 318):
        if n % 16:
            a = random_dna(rng, 900)
            As.append(a)
            Bs.append(random_dna(rng, n - 50) + a[400:450])        # the best local alignment ends at (450, n)
    h = bx.largest_h(900, 317, 0, bx.span)
    assert 16 * h > 1 << 30
    wants = [po.align(a, b, 0, h, mode=po.LOCAL) for a, b in zip(As, Bs)]
    assert all((w.end_j - 1) // 16 == (len(b) - 1) // 16 for w, b in zip(wants, Bs))
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    routes = [("banded", ctx.align_batch_banded(ba, oa, la, bb, ob, lb, 900, psa.LOCAL, 0, h, traceback=False)[0]),
              ("banded_device", batch_device(ctx, As, Bs, 900, psa.LOCAL, 0, h, False)[0])]
    generic = psa.Context(0)
    generic.set_option("pack", 0)
    routes.append(("long_batch", generic.align_batch(ba, oa, la, bb, ob, lb, psa.LOCAL, 0, h, traceback=False)[0]))
    generic.close()
    for name, items in routes:
        for k, w in enumerate(wants):
            assert (int(items[k]["score"]), int(items[k]["end_i"]), int(items[k]["end_j"])) == (w.score, w.end_i, w.end_j), (name, k)
    for geo in (2, 3):
        c = psa.Context(0)
        c.set_option("long_geometry", geo)
        for k, w in enumerate(wants):
            r = c.align_pair(As[k], Bs[k], psa.LOCAL, 0, h, traceback=False)
            assert (r.score, r.end_i, r.end_j) == (w.score, w.end_i, w.end_j), (geo, k)
        c.close()


# ---- (d) a band that holds every cell keeps the unbanded limit and equals the unbanded entries ----------------

@pytest.mark.parametrize("mode", MODES)
def test_wide_band_at_the_unbanded_limit(ctx, mode):
    import torch
    from tests.test_gpu_banded_pair import Dev
    for m, n, related in ((300, 900, False), (900, 300, False), (1000, 1040, True)):
        a, b = edge_pair(m, n, related, m + n)
        ba, oa, la = psa.pack_pairs([a])
        bb, ob, lb = psa.pack_pairs([b])
        for g, h in ((0, bx.largest_h(m, n, 0, bx.span)), (bx.largest_g(m, n, 0, bx.span), 0),
                     (bx.largest_g(m, n, 1, bx.span), 1)):
            for band in (max(m, n), max(m, n) + 5):
                tag = (m, n, g, h, band)
                for tb in (True, False):
                    ref_items, ref_ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=tb)
                    items, ops = ctx.align_batch_banded(ba, oa, la, bb, ob, lb, band, mode, g, h, traceback=tb)
                    ditems, dops = batch_device(ctx, [a], [b], band, mode, g, h, tb)
                    assert items.tobytes() == ref_items.tobytes() == ditems.tobytes(), (tag, tb)
                    nw = (int(ref_items[0]["aln_len"]) + 15) // 16
                    if tb:
                        assert np.array_equal(ops[0, :nw], ref_ops[0, :nw]) and np.array_equal(dops[0, :nw], ref_ops[0, :nw]), tag
                    want, got = ctx.align_pair(a, b, mode, g, h, traceback=tb), ctx.align_pair_banded(a, b, band, mode, g, h, traceback=tb)
                    for f in ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j", "start_i", "start_j", "ops", "row_a", "row_b"):
                        assert getattr(got, f) == getattr(want, f), (tag, tb, f)
                    st = torch.cuda.Stream()
                    ref, banded = Dev(a, b, st), Dev(a, b, st)
                    ref.run(ctx, 0, mode, g, h, tb=tb, banded=False)
                    banded.run(ctx, band, mode, g, h, tb=tb)
                    st.synchronize()
                    (ri, ro), (bi, bo_) = ref.result(), banded.result()
                    assert bi.tobytes() == ri.tobytes() and np.array_equal(bo_[:nw], ro[:nw]), (tag, tb)
                over = (g, h + 1) if g == 0 else (g + 1, h)
                expect_range_error(ctx, a, b, band, mode, *over, tag=tag)


# ---- (e) no path in the band, at the limit -------------------------------------------------------------------

def test_no_path_record_at_the_limit(ctx):
    for m, n, band in ((2, 1000, 10), (40, 8000, 10), (1, 500, 3)):
        assert n > (2 * band + 1) * m
        a, b = edge_pair(m, n, False, n)
        for (g, h), _ in edge_penalties(m, n):
            w = check(ctx, a, b, band, psa.GLOBAL, g, h, tag=(m, n))
            assert (w.t1, w.t2, w.t3, w.score, w.end_state, w.ops) == (NEG_INF, NEG_INF, NEG_INF, NEG_INF, 1, b"")
