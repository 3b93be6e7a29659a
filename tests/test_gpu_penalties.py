"""Every kernel family against the oracle at gap penalties other than (g, h) = (1, 2).

Each family folds g and h into constants of its own (biases, packed (-g, -g) / (g+h, g+h) pairs, byte tables, the
crossing rule Ff + Fr + h).  At (1, 2) h == 2g, h == g + 1 and 2h == g + h + 1, so a g where an h belongs, or an h
where 2g belongs, gives the right answer there.  The grid below keeps g, h, g+h, 2g, 2h and h-g apart where it can, and
adds the degenerate settings.  Beyond it: the largest g the packed kernels' 16-bit envelopes admit (and g + 1, which
must leave the packed path and still be right), and the largest penalties the int32 kernels admit, where untyped
corners come within a few thousand of -2^28 and typed ones (three gap openings) reach -3h.  Every comparison is
exact."""
import functools
import random

import numpy as np
import pytest

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200 import synth
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
from oracle import pyoracle as po
from tests.helpers import mutated_copy, py_random_pair, random_dna

pytestmark = pytest.mark.gpu

GRID = [(0, 0), (0, 1), (2, 0), (3, 1), (5, 2)]          # every family (the packed short kernel takes h <= 2)
WIDE = GRID + [(1, 7), (4, 9), (0, 11)]                    # families without the h <= 2 limit
ERR_RANGE = -2
SPAN_LIMIT = 1 << 28


# ---- mirrors of the dispatch predicates (csrc/psa_pack.cu, csrc/psa_pack_long.cu, csrc/psa_capi.cu) ----

def pack_bias(mode, g, h, m, n):
    decay = g * (m + n) + 2 * (g + h)
    if mode == psa.LOCAL:
        return (g + h) + 16 + decay
    return g * (m + n) + 2 * h + (g + h) + 16 + decay


def pack_supported(m, n, mode, g, h):
    """psa_pack_supported: the .S16x2 short-read kernel."""
    if not (1 <= m <= 512 and 1 <= n <= 256) or h > 2 or g + h + 1 > 120:
        return False
    if mode == psa.LOCAL and g + h < 1:
        return False
    top = pack_bias(mode, g, h, m, n) + min(m, n) + g + h + 2
    return top * 32 + 31 < 65536 if mode == psa.LOCAL else top < 32000


def pack_long_supported(m, n, mode, g, h):
    """psa_pack_long_supported: the .S16x2 strip kernel for batches of long pairs."""
    if m < 1 or n < 1 or g + h + 1 > 120:
        return False
    if mode == psa.LOCAL and g + h < 1:
        return False
    mn = min(m, n)
    if mode == psa.LOCAL:
        return (g + h + 16 + mn) * 8 + 7 < 65536
    return g * (m + n) + 2 * h + (g + h) + 16 + mn + g + h + 2 < 32700


def largest_g(pred, h):
    g = 0
    while pred(g + 1, h):
        g += 1
    assert pred(g, h)
    return g


def int32_limits(m, n):
    """check_scoring: g (m + n + 2) + 2h + m + n < 2^28.  Largest h at g = 0, largest g at h = 0 and at h = 1."""
    free = SPAN_LIMIT - 1 - m - n
    return [(0, free // 2), (free // (m + n + 2), 0), ((free - 2) // (m + n + 2), 1)]


def span(g, h, m, n):
    return g * (m + n + 2) + 2 * h + m + n


# ---- oracle, cached: several routes are compared with the same answers ----

@functools.lru_cache(maxsize=None)
def aln(a, b, g, h, mode=po.GLOBAL, st=-1, et=-1):
    return po.align(a, b, g, h, mode=mode, start_type=st, end_type=et)


@functools.lru_cache(maxsize=None)
def lin(a, b, g, h, mode=po.GLOBAL):
    return po.score_linear(a, b, g, h, mode=mode)


def same_score(it, want, mode, tag):
    """Batch record (or PairResult) vs oracle: score, end cell; corners and end state in global mode."""
    get = (lambda f: it[f]) if isinstance(it, np.void) else (lambda f: getattr(it, f))
    assert get("score") == want.score, tag
    assert (get("end_i"), get("end_j")) == (want.end_i, want.end_j), tag
    if mode == psa.GLOBAL:
        assert (get("t1"), get("t2"), get("t3"), get("end_state")) == (want.t1, want.t2, want.t3, want.end_state), tag


def same_aln(it, words, a, b, want, mode, tag):
    """Batch record + op words vs the oracle's full alignment, rows included."""
    same_score(it, want, mode, tag)
    assert (it["start_i"], it["start_j"]) == (want.start_i, want.start_j), tag
    ops = psa.unpack_ops(words, int(it["aln_len"]))
    assert ops == want.ops, tag
    assert psa.render_rows(a, b, ops, int(it["start_i"]), int(it["start_j"])) == (want.row_a, want.row_b), tag


def same_pair(got, want, mode, tag):
    same_score(got, want, mode, tag)
    assert (got.start_i, got.start_j) == (want.start_i, want.start_j), tag
    assert got.ops == want.ops and (got.row_a, got.row_b) == (want.row_a, want.row_b), tag


def same_records(items, ops, ref_items, ref_ops, tag):
    """Two routes, byte-identical: every item field and every op word that carries ops."""
    for f in ITEM_DTYPE.names:
        assert np.array_equal(items[f], ref_items[f]), (tag, f, np.flatnonzero(items[f] != ref_items[f])[:8])
    if ops is not None:
        words = (items["aln_len"].astype(np.int64) + 15) // 16
        mask = np.arange(ops.shape[1])[None, :] < words[:, None]
        assert np.array_equal(ops[mask], ref_ops[mask]), tag


def check_empty(it, a, b, g, h, mode, tag):
    assert it["aln_len"] == 0, tag
    if mode == psa.GLOBAL:
        w = po.score_linear(a, b, g, h)
        assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (w.t1, w.t2, w.t3, w.end_state), tag
    else:
        assert (it["score"], it["end_i"], it["end_j"]) == (0, 0, 0), tag


def batch(ctx, As, Bs, mode, g, h, tb):
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    l0 = ctx.launches
    items, ops = ctx.align_batch(ba, oa, la, bb, ob, lb, mode, g, h, traceback=tb)
    return items, ops, ctx.launches - l0


def new_ctx(**options):
    c = psa.Context(0)
    for k, v in options.items():
        c.set_option(k, v)
    return c


@pytest.fixture(scope="module")
def ctx():
    c = psa.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def generic():
    """The int32 kernels only (pack = 0): the second route of every packed comparison."""
    c = new_ctx(pack=0)
    yield c
    c.close()


# ---- 1. packed short fill and walks ----------------------------------------------------------------------------

# (max m, max n): one batch per (G, K) instantiation of pick_shape, and m up to 512
SHORT_SHAPES = [(32, 32), (70, 64), (96, 96), (140, 128), (150, 150), (160, 160), (200, 192), (512, 256)]


@functools.lru_cache(maxsize=None)
def short_batch(max_m, max_n):
    """72 ragged pairs with both maxima present.  Pairs 10-15 put members with m = 1 or n = 1 next to full-size members
    in the same pair-of-pairs (indices 2q, 2q+1): their padding cells are what the second g(m+n) of pack_bias covers.
    From 16 on, members the packed fill must flag (N, lower case, empty, another alphabet)."""
    rnd = random.Random(max_m * 1000 + max_n)
    rng = np.random.default_rng(max_m * 1000 + max_n)
    pairs = []
    for k in range(72):
        a, b = py_random_pair(rnd, max_m, max_n, b"ACGT")
        b = b[:max_n]
        if k >= 16 and k % 23 == 5:
            a = a.replace(b"A", b"N")
        if k >= 16 and k % 29 == 7:
            b = b.lower()
        if k >= 16 and k % 31 == 9:
            a = b""
        if k >= 16 and k % 37 == 11:
            a, b = py_random_pair(rnd, max_m, max_n, b"ABCDEFGHIJKLMNOPQRSTUVWY")
            b = b[:max_n]
        pairs.append((a, b))

    def full():
        a = random_dna(rng, max_m)
        return a, mutated_copy(rng, a, max_n)

    pairs[10], pairs[11] = full(), (random_dna(rng, 1), random_dna(rng, max_n))
    pairs[12], pairs[13] = (random_dna(rng, max_m), random_dna(rng, 1)), full()
    pairs[14], pairs[15] = full(), (random_dna(rng, 1), random_dna(rng, 1))
    As, Bs = [p[0] for p in pairs], [p[1] for p in pairs]
    assert max(map(len, As)) == max_m and max(map(len, Bs)) == max_n
    return As, Bs


def check_short(As, Bs, items, ops, g, h, mode, tag):
    for k, (a, b) in enumerate(zip(As, Bs)):
        if not a or not b:
            check_empty(items[k], a, b, g, h, mode, (tag, k))
        elif ops is not None:
            same_aln(items[k], ops[k], a, b, aln(a, b, g, h, mode), mode, (tag, k))
        else:
            same_score(items[k], aln(a, b, g, h, mode), mode, (tag, k))


def packed_launches(tb, flavour):
    """Launches of a one-chunk packed batch: fill, walk (codes: 1; checkpoints: 2 perm passes + walk), flagged members."""
    return 2 + (0 if not tb else (3 if flavour else 1))


@pytest.mark.parametrize("shape", SHORT_SHAPES, ids=[f"{m}x{n}" for m, n in SHORT_SHAPES])
def test_packed_short_grid(shape):
    """Both traceback flavours, traceback on and off, both modes, the grid; packed whenever the predicate admits it."""
    As, Bs = short_batch(*shape)
    ctxs = {f: new_ctx(pack_traceback=f) for f in (0, 1)}
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            for g, h in GRID:
                packed = pack_supported(shape[0], shape[1], mode, g, h)
                for flavour, c in ctxs.items():
                    for tb in (True, False):
                        tag = (shape, mode, g, h, flavour, tb)
                        items, ops, launches = batch(c, As, Bs, mode, g, h, tb)
                        assert launches == (packed_launches(tb, flavour) if packed else 1), tag
                        check_short(As, Bs, items, ops, g, h, mode, tag)
    finally:
        for c in ctxs.values():
            c.close()


def packed_entry_accepts(ctx, m, n, mode, g, h):
    """psa_align_batch_packed returns PSA_ERR_RANGE exactly where psa_pack_supported is false (score only: the short-read
    envelope holds for both traceback settings at these shapes)."""
    a2 = psa.pack_reads_2bit(np.frombuffer(b"ACGT" * 128, dtype=np.uint8)[:m].reshape(1, m))
    b2 = psa.pack_reads_2bit(np.frombuffer(b"CGTA" * 64, dtype=np.uint8)[:n].reshape(1, n))
    try:
        ctx.align_batch_packed(a2, b2, m, n, mode, g, h, traceback=False)
        return True
    except psa.PsaError as e:
        assert e.code == ERR_RANGE
        return False


@pytest.mark.parametrize("shape", SHORT_SHAPES, ids=[f"{m}x{n}" for m, n in SHORT_SHAPES])
def test_packed_short_largest_g(ctx, shape):
    """At each shape, mode and h in {0, 2}: the largest g the 16-bit envelope admits runs packed; g + 1 runs the int32
    kernel.  Both equal the oracle.  The library's own predicate must agree with the mirror at both."""
    As, Bs = short_batch(*shape)
    m, n = shape
    for mode in (psa.GLOBAL, psa.LOCAL):
        for h in (0, 2):
            gmax = largest_g(lambda g, hh: pack_supported(m, n, mode, g, hh), h)
            assert packed_entry_accepts(ctx, m, n, mode, gmax, h), (shape, mode, gmax, h)
            assert not packed_entry_accepts(ctx, m, n, mode, gmax + 1, h), (shape, mode, gmax + 1, h)
            for g in (gmax, gmax + 1):
                for tb in (True, False):
                    tag = (shape, mode, g, h, tb)
                    items, ops, launches = batch(ctx, As, Bs, mode, g, h, tb)
                    assert launches == (packed_launches(tb, 0) if g == gmax else 1), tag
                    check_short(As, Bs, items, ops, g, h, mode, tag)


# ---- 2. the 2-bit entry and the byte-input host pipeline --------------------------------------------------------

@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_packed_2bit_entry(generic, mode):
    """psa_align_batch_packed over several 1 024-pair chunks == the byte entry through the int32 kernel, at two grid
    settings and at the largest g the 150 x 150 envelope admits."""
    m, n, npairs = 150, 150, 2100
    A, _ = synth.read_pair_batch(npairs, m, 4100 + mode)
    rng = np.random.default_rng(4200 + mode)
    B = synth.ACGT[synth.random_codes(rng, npairs, n)]
    B[0::2] = A[0::2]
    mut = rng.random((npairs, n)) < 0.08
    B[mut] = synth.ACGT[rng.integers(0, 4, size=int(mut.sum()))]
    a2, b2 = psa.pack_reads_2bit(A), psa.pack_reads_2bit(B)
    offa, la = synth.fixed_length_layout(npairs, m)
    offb, lb = synth.fixed_length_layout(npairs, n)
    c = new_ctx(pack_chunk=1024)
    try:
        gmax = largest_g(lambda g, hh: pack_supported(m, n, mode, g, hh), 0)
        for g, h in [(3, 1), (5, 2), (gmax, 0)]:
            for tb in (True, False):
                tag = (mode, g, h, tb)
                items, ops = c.align_batch_packed(a2, b2, m, n, mode, g, h, traceback=tb)
                ref, ref_ops = generic.align_batch(A.reshape(-1), offa, la, B.reshape(-1), offb, lb, mode, g, h, traceback=tb)
                for f in ("score", "end_i", "end_j", "end_state") + (("start_i", "start_j", "aln_len") if tb else ()):
                    assert np.array_equal(items[f].astype(np.int64), ref[f].astype(np.int64)), (tag, f)
                if tb:
                    words = (ref["aln_len"].astype(np.int64) + 15) // 16
                    mask = np.arange(ops.shape[1])[None, :] < words[:, None]
                    assert np.array_equal(ops[mask], ref_ops[:, :ops.shape[1]][mask]), tag
                for q in range(0, npairs, 211):
                    w = aln(A[q].tobytes(), B[q].tobytes(), g, h, mode)
                    assert (items[q]["score"], items[q]["end_i"], items[q]["end_j"]) == (w.score, w.end_i, w.end_j), (tag, q)
                    if tb:
                        assert psa.unpack_ops(ops[q], int(items[q]["aln_len"])) == w.ops, (tag, q)
        with pytest.raises(psa.PsaError) as e:
            c.align_batch_packed(a2, b2, m, n, mode, gmax + 1, 0, traceback=False)
        assert e.value.code == ERR_RANGE
    finally:
        c.close()


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_byte_pipeline(mode):
    """psa_align_batch through the chunked host pipeline (> 1 024 contiguous pairs, 1 024-pair chunks) == pipeline = 0,
    flagged members included, at two grid settings; a sample == the oracle.  The pipeline plans its constants once per
    call, so a stale default would show here."""
    n = 2600
    rng = np.random.default_rng(2600 + mode)
    la, lb = rng.integers(1, 151, size=n), rng.integers(1, 151, size=n)
    la[0], lb[0] = 150, 150
    As = [random_dna(rng, int(x)) for x in la]
    Bs = [mutated_copy(rng, a, int(y)) if k % 2 else random_dna(rng, int(y)) for k, (a, y) in enumerate(zip(As, lb))]
    for j, q in enumerate(range(7, n, 401)):
        if j % 3 == 0:
            As[q] = As[q][:-1] + b"N"
        elif j % 3 == 1:
            Bs[q] = Bs[q].lower()
        else:
            As[q] = b""
    chunks = -(-n // 1024)
    c = new_ctx(pack_chunk=1024)
    try:
        for g, h in [(3, 1), (5, 2)]:
            for tb in (True, False):
                tag = (mode, g, h, tb)
                c.set_option("pipeline", 1)
                items, ops, launches = batch(c, As, Bs, mode, g, h, tb)
                assert launches == chunks * packed_launches(tb, 0), tag
                c.set_option("pipeline", 0)
                ref, ref_ops, _ = batch(c, As, Bs, mode, g, h, tb)
                same_records(items, ops, ref, ref_ops, tag)
                for q in list(range(0, n, 97)) + list(range(7, n, 401)):
                    if As[q] and Bs[q]:
                        w = aln(As[q], Bs[q], g, h, mode)
                        if tb:
                            same_aln(items[q], ops[q], As[q], Bs[q], w, mode, (tag, q))
                        else:
                            same_score(items[q], w, mode, (tag, q))
                    else:
                        check_empty(items[q], As[q], Bs[q], g, h, mode, (tag, q))
    finally:
        c.close()


# ---- 3. packed long batches (.S16x2 strips) and 4. the int32 long batch ------------------------------------------

def long_batch_pairs(seed, count, lo, hi, odd_member=True):
    rng = np.random.default_rng(seed)
    As, Bs = [], []
    for k in range(count):
        m, n = int(rng.integers(lo, hi + 1)), int(rng.integers(lo, hi + 1))
        a = random_dna(rng, m)
        As.append(a)
        Bs.append(mutated_copy(rng, a, n) if k % 3 else random_dna(rng, n))
    if odd_member:
        As[3] = As[3][:100] + b"N" + As[3][101:]          # not plain ACGT: the int32 kernel recomputes it
    return As, Bs


def check_long_scores(As, Bs, items, g, h, mode, tag):
    for k, (a, b) in enumerate(zip(As, Bs)):
        if not a or not b:
            check_empty(items[k], a, b, g, h, mode, (tag, k))
        else:
            same_score(items[k], lin(a, b, g, h, mode), mode, (tag, k))


LOCAL_WIDE_EXTRA = [(119, 0), (7, 112), (120, 0)]     # g + h = 119 is the packed long kernel's last; 120 is not packed


@pytest.mark.parametrize("k", [8, 16])
@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_packed_long_grid(generic, mode, k):
    """11 pairs (an odd count, one non-ACGT member), lane width forced to 8 and 16 columns: the grid including h > 2,
    and in local mode g + h = 119 and 120.  == the linear-space oracle, and == pack = 0 byte for byte."""
    As, Bs = long_batch_pairs(3000 + mode, 11, 300, 1500)
    c = new_ctx(pack_long_k=k)
    try:
        for g, h in WIDE + (LOCAL_WIDE_EXTRA if mode == psa.LOCAL else []):
            tag = (mode, k, g, h)
            packed = pack_long_supported(max(map(len, As)), max(map(len, Bs)), mode, g, h)
            items, _, launches = batch(c, As, Bs, mode, g, h, False)
            assert launches == (2 if packed else 1), tag
            check_long_scores(As, Bs, items, g, h, mode, tag)
            ref, _, _ = batch(generic, As, Bs, mode, g, h, False)
            same_records(items, None, ref, None, tag)
    finally:
        c.close()


@pytest.mark.parametrize("size", [800, 1200])
def test_packed_long_largest_global_g(ctx, generic, size):
    """Global mode at the largest g the packed long kernel admits for size^2 pairs (and g + 1, int32), h = 0 and 2."""
    rng = np.random.default_rng(size)
    As = [random_dna(rng, size) for _ in range(9)]
    Bs = [mutated_copy(rng, a, size) if k % 2 else random_dna(rng, size) for k, a in enumerate(As)]
    for h in (0, 2):
        gmax = largest_g(lambda g, hh: pack_long_supported(size, size, psa.GLOBAL, g, hh), h)
        for g in (gmax, gmax + 1):
            tag = (size, g, h)
            items, _, launches = batch(ctx, As, Bs, psa.GLOBAL, g, h, False)
            assert launches == (2 if g == gmax else 1), tag
            check_long_scores(As, Bs, items, g, h, psa.GLOBAL, tag)
            ref, _, _ = batch(generic, As, Bs, psa.GLOBAL, g, h, False)
            same_records(items, None, ref, None, tag)


@pytest.mark.parametrize("mode,size", [(psa.LOCAL, 8172), (psa.GLOBAL, 10890)])
def test_packed_long_identical_copy_at_the_bound(ctx, generic, mode, size):
    """An identical pair at the largest size the 16-bit lanes admit at (1, 2): in local mode the key (T1 + bias) * 8 + 7
    reaches exactly 65 535; in global mode the corner sits at the top of the biased range.  One size more is refused."""
    assert pack_long_supported(size, size, mode, 1, 2) and not pack_long_supported(size + 1, size + 1, mode, 1, 2)
    if mode == psa.LOCAL:
        assert (size + 1 + 2 + 16) * 8 + 7 == 65535
    rng = np.random.default_rng(size)
    a = random_dna(rng, size)
    As = [a] + [random_dna(rng, int(rng.integers(300, 900))) for _ in range(8)]
    Bs = [a] + [mutated_copy(rng, x, len(x) + 20) for x in As[1:]]
    items, _, launches = batch(ctx, As, Bs, mode, 1, 2, False)
    assert launches == 2
    check_long_scores(As, Bs, items, 1, 2, mode, (mode, size))
    assert items[0]["score"] == size
    ref, _, _ = batch(generic, As, Bs, mode, 1, 2, False)
    same_records(items, None, ref, None, (mode, size))


@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_int32_long_batch_score_only(generic, mode):
    """pack = 0: the int32 one-warp-per-pair batch kernel, ragged lengths 300 - 2 000 and empty members, the grid."""
    As, Bs = long_batch_pairs(5000 + mode, 14, 300, 2000, odd_member=False)
    rng = np.random.default_rng(5100 + mode)
    As += [b"", random_dna(rng, 400)]
    Bs += [random_dna(rng, 400), b""]
    for g, h in WIDE:
        items, _, launches = batch(generic, As, Bs, mode, g, h, False)
        assert launches == 1
        check_long_scores(As, Bs, items, g, h, mode, (mode, g, h))


# ---- 5. one long pair --------------------------------------------------------------------------------------------

TILE_EDGE_SHAPES = [(129, 257), (255, 513), (383, 769)]     # across the 128-row and 256-column tile edges


@functools.lru_cache(maxsize=None)
def long_pairs(shapes, seed):
    rng = np.random.default_rng(seed)
    out = []
    for k, (m, n) in enumerate(shapes):
        a = random_dna(rng, m)
        out.append((a, mutated_copy(rng, a, n) if k % 2 == 0 else random_dna(rng, n)))
    return out


@pytest.mark.parametrize("band", [1, 0])
@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_long_single_traceback(mode, band):
    """Checkpointed fill + traceback of one pair, the grid, with the ahead-of-time band recompute (long_band = 1, the
    default) and without it (each tile recomputed on demand by the walk)."""
    pairs = long_pairs(tuple(TILE_EDGE_SHAPES + [(1000, 1030), (2000, 2100)]), 55)
    c = new_ctx(long_band=band)
    try:
        for g, h in WIDE:
            for a, b in pairs:
                same_pair(c.align_pair(a, b, mode, g, h), aln(a, b, g, h, mode), mode, (mode, band, g, h, len(a), len(b)))
    finally:
        c.close()


@pytest.mark.parametrize("geo", [-1, 6, 7, 2, 0])
def test_long_single_score_only(geo):
    """Score-only fill of one pair on the default geometry and on the forced tile geometries 6, 7, 2 and 0."""
    pairs = long_pairs(((700, 1500), (1300, 2100)), 66)
    c = new_ctx(long_geometry=geo)
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            for g, h in WIDE:
                for a, b in pairs:
                    got = c.align_pair(a, b, mode, g, h, traceback=False)
                    same_score(got, lin(a, b, g, h, mode), mode, (geo, mode, g, h, len(a)))
    finally:
        c.close()


# ---- 6. the systolic kernel --------------------------------------------------------------------------------------

@pytest.mark.parametrize("kc", [8, 4])
def test_systolic_kernel(kc):
    """long_systolic = 1 (the kernel serves score-only calls), 8 and 4 columns per lane: small pairs and one
    6 k x 9 k pair, the grid, both modes."""
    pairs = long_pairs(((300, 700), (129, 2049), (6000, 9000)), 77)
    c = new_ctx(long_systolic=1, systolic_kc=kc)
    assert c.long_strip_columns == 32 * kc
    try:
        for mode in (psa.GLOBAL, psa.LOCAL):
            for g, h in WIDE:
                for a, b in pairs:
                    got = c.align_pair(a, b, mode, g, h, traceback=False)
                    same_score(got, lin(a, b, g, h, mode), mode, (kc, mode, g, h, len(a)))
    finally:
        c.close()


# ---- 7. batches of long pairs with traceback ---------------------------------------------------------------------

def device_batch(ctx, As, Bs, mode, g, h):
    """psa_align_batch_device with traceback, on a torch side stream."""
    import torch
    dev = torch.device("cuda", 0)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    n = len(As)
    stride = (int(la.max()) + int(lb.max()) + 15) // 16 + 1
    st = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(st):
        pad = np.zeros(1, dtype=np.uint8)
        t = [torch.from_numpy(x).to(dev) for x in (np.concatenate([ba, pad]), oa, la, np.concatenate([bb, pad]), ob, lb)]
        items = torch.zeros(n * 10, dtype=torch.int32, device=dev)
        ops = torch.zeros(n * stride, dtype=torch.int32, device=dev)
        st.synchronize()
        ctx.align_batch_device(*(x.data_ptr() for x in t), n, int(la.max()), int(lb.max()), items.data_ptr(), ops.data_ptr(),
                               stride, mode, g, h, True, st.cuda_stream)
        st.synchronize()
    return items.cpu().numpy().view(ITEM_DTYPE).copy(), ops.cpu().numpy().view(np.uint32).reshape(n, stride).copy()


@pytest.mark.parametrize("gh", [(0, 0), (3, 1), (5, 2), (0, 11)])
@pytest.mark.parametrize("mode", [psa.GLOBAL, psa.LOCAL])
def test_long_batch_traceback(ctx, mode, gh):
    """20 ragged long pairs (the batched fill + walk), through the host and the device entry."""
    g, h = gh
    As, Bs = long_batch_pairs(7000 + 10 * mode + g, 20, 257, 1500, odd_member=False)
    hi, ho, _ = batch(ctx, As, Bs, mode, g, h, True)
    di, do = device_batch(ctx, As, Bs, mode, g, h)
    same_records(hi, ho, di, do, (mode, g, h))
    for k in range(len(As)):
        same_aln(hi[k], ho[k], As[k], Bs[k], aln(As[k], Bs[k], g, h, mode), mode, (mode, g, h, k))


# ---- 8. the partition finder -------------------------------------------------------------------------------------

def rescore_rows(row_a, row_b, g, h):
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
def test_partition_finder(ctx, pieces):
    """align_long_partitioned at the grid: a complete alignment that re-scores, with the same g and h, to the oracle's
    optimum; crossings on special rows."""
    pairs = long_pairs(((1000, 1100), (3000, 2500), (2049, 300)), 88)
    for g, h in WIDE:
        for a, b in pairs:
            tag = (pieces, g, h, len(a), len(b))
            got, crossings = ctx.align_long_partitioned(a, b, pieces, g, h)
            want = lin(a, b, g, h)
            assert got.score == want.score, tag
            assert got.row_a.replace(b"-", b"") == a and got.row_b.replace(b"-", b"") == b, tag
            assert rescore_rows(got.row_a, got.row_b, g, h) == want.score, tag
            assert len(crossings) <= pieces - 1 and crossings == sorted(crossings), tag
            assert all(i % 128 == 0 and 0 < i < len(a) and 0 <= j <= len(b) and t in (1, 3) for i, j, t in crossings), tag
            if pieces > 2 and g + h > 0:
                assert len(crossings) >= 1, tag


def test_partition_finder_gap_across_the_special_row(ctx):
    """A = B with 300 extra bases in A across the row the finder picks for two pieces.  The optimal path crosses that
    row inside a vertical gap: for h > 0 the gap's value Ff + Fr + h beats the node's Hf + Hr by h, so the crossing has
    type 3; for h = 0 the two tie and the node (type 1) wins by priority."""
    rng = np.random.default_rng(300)
    b = random_dna(rng, 2000)
    a = b[:1000] + random_dna(rng, 300) + b[1000:]
    avail = (len(a) - 1) // 128
    row = (avail + 1) // 2 * 128                           # the one special row of a two-piece call
    assert 1000 < row < 1300
    for g, h in WIDE:
        tag = (g, h)
        got, crossings = ctx.align_long_partitioned(a, b, 2, g, h)
        want = lin(a, b, g, h)
        assert got.score == want.score and rescore_rows(got.row_a, got.row_b, g, h) == want.score, tag
        if (g, h) != (0, 0):                               # without any gap cost, ties may leave the cut out
            assert len(crossings) == 1, (tag, crossings)
        for i, j, t in crossings:
            assert i == row and t == (3 if h > 0 else 1), (tag, crossings)


# ---- 9. the int32 kernels at the edge of check_scoring -----------------------------------------------------------

def corners_near_the_limit(results, below=-(1 << 27)):
    """The cases must reach below `below`: finite corners down there are what out_value's threshold must keep finite."""
    finite = [v for r in results for v in (r.t1, r.t2, r.t3) if v != psa.capi.NEG_INF]
    assert min(finite) < below


@pytest.mark.parametrize("shape", [(150, 150), (300, 700)], ids=["short", "long_single"])
def test_int32_range_limit_single_pair(ctx, shape):
    """align_pair at the largest h (g = 0) and the largest g (h = 0 and 1) that check_scoring admits, plus typed
    start / end types; one more is PSA_ERR_RANGE."""
    m, n = shape
    rng = np.random.default_rng(m + n)
    a = random_dna(rng, m)
    b = mutated_copy(rng, a, n)
    wants = []
    for g, h in int32_limits(m, n):
        assert span(g, h, m, n) < SPAN_LIMIT
        for mode in (psa.GLOBAL, psa.LOCAL):
            want = aln(a, b, g, h, mode)
            same_pair(ctx.align_pair(a, b, mode, g, h), want, mode, (shape, mode, g, h))
            got = ctx.align_pair(a, b, mode, g, h, traceback=False)
            same_score(got, want, mode, (shape, mode, g, h, "score only"))
            wants.append(want)
        for st, et in ((-2, -3), (-3, 2), (2, -2), (3, 3), (1, -1)):
            want = aln(a, b, g, h, po.GLOBAL, st, et)
            same_pair(ctx.align_pair(a, b, psa.GLOBAL, g, h, start_type=st, end_type=et), want, psa.GLOBAL, (shape, g, h, st, et))
            wants.append(want)
        over = (g, h + 1) if g == 0 else (g + 1, h)
        assert span(*over, m, n) >= SPAN_LIMIT
        with pytest.raises(psa.PsaError) as e:
            ctx.align_pair(a, b, psa.GLOBAL, *over)
        assert e.value.code == ERR_RANGE
    corners_near_the_limit(wants, -(1 << 28))    # typed corners with three gap openings: about -3h


def test_int32_range_limit_long_batches(ctx):
    """16 long pairs up to 300 x 700: the batched traceback path and the score-only batch (the packed long kernel
    refuses these penalties), at the int32 limits; then typed pieces through psa_align_partition, 17 pieces wider
    than 256 columns (the batched traceback path)."""
    rng = np.random.default_rng(1600)
    As, Bs = [random_dna(rng, 300)], [None]
    Bs[0] = mutated_copy(rng, As[0], 700)
    for k in range(15):
        a = random_dna(rng, int(rng.integers(257, 301)))
        As.append(a)
        Bs.append(mutated_copy(rng, a, int(rng.integers(257, 701))) if k % 2 else random_dna(rng, int(rng.integers(257, 701))))
    wants = []
    for g, h in int32_limits(300, 700):
        assert not pack_long_supported(300, 700, psa.GLOBAL, g, h)
        for mode in (psa.GLOBAL, psa.LOCAL):
            tag = (mode, g, h)
            items, ops, _ = batch(ctx, As, Bs, mode, g, h, True)
            scores, _, launches = batch(ctx, As, Bs, mode, g, h, False)
            assert launches == 1, tag
            for k in range(len(As)):
                want = aln(As[k], Bs[k], g, h, mode)
                same_aln(items[k], ops[k], As[k], Bs[k], want, mode, (tag, k))
                same_score(scores[k], want, mode, (tag, k, "score only"))
                wants.append(want)
        over = (g, h + 1) if g == 0 else (g + 1, h)
        for tb in (True, False):
            with pytest.raises(psa.PsaError) as e:
                batch(ctx, As, Bs, psa.GLOBAL, *over, tb)
            assert e.value.code == ERR_RANGE
    corners_near_the_limit(wants)

    a = random_dna(rng, 17 * 290)
    b = mutated_copy(rng, a, 17 * 300)
    types = [-3, -2, -1, 1, 2, 3]
    points = [(0, 0, -1)] + [(k * 290, k * 300 + int(rng.integers(-5, 6)), types[k % 6]) for k in range(1, 17)] + [(len(a), len(b), 1)]
    pm = max(i1 - i0 for (i0, _, _), (i1, _, _) in zip(points[:-1], points[1:]))
    pn = max(j1 - j0 for (_, j0, _), (_, j1, _) in zip(points[:-1], points[1:]))
    assert min(j1 - j0 for (_, j0, _), (_, j1, _) in zip(points[:-1], points[1:])) > 256
    wants = []
    for g, h in int32_limits(pm, pn):
        ops = ra = rb = b""
        for (i0, j0, t0), (i1, j1, t1) in zip(points[:-1], points[1:]):
            piece = aln(a[i0:i1], b[j0:j1], g, h, po.GLOBAL, t0, -t1)
            ops += piece.ops; ra += piece.row_a; rb += piece.row_b
            wants.append(piece)
        got = ctx.align_partition(a, b, points, g, h)
        assert (got.ops, got.row_a, got.row_b) == (ops, ra, rb), (g, h)
        assert (got.t1, got.t2, got.t3, got.end_state) == (piece.t1, piece.t2, piece.t3, piece.end_state), (g, h)
        over = (g, h + 1) if g == 0 else (g + 1, h)
        with pytest.raises(psa.PsaError) as e:
            ctx.align_partition(a, b, points, *over)
        assert e.value.code == ERR_RANGE
    corners_near_the_limit(wants)
