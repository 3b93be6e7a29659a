"""The band of an anchor chain (psa_align_batch_guided, include/psa.h) on the CPU: guide_rows against the diagonal band
for an empty chain, the properties the kernels rely on for random valid chains (monotone rows, the checkpoint bound of
banded_slot_bytes), the per-row oracles against the banded ones and the exact reference, and the int32 arithmetic of the
kernels at the edge of check_banded_scoring on chains that force a gap opening on every row.  No GPU."""
import random

import numpy as np
import pytest

from oracle import pyoracle as po
from tests import banded_exact as bx
from tests import banded_oracle as bo
from tests import guided_exact as gx
from tests import guided_oracle as go
from tests.helpers import mutated_copy, py_random_pair, random_dna
from tests.test_banded_range_cpu import CUT, KNEG, edge_penalties, exact_record, w32

R, W = 128, 256
RECORD = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j")


def random_chain(rnd, m, n, k):
    """A valid chain of k anchors: independent sorted coordinates (so duplicates and runs occur), with some forced
    onto rows 0 / m and columns 0 / n and some long horizontal and vertical runs."""
    if k == 0:
        return np.zeros((0, 2), dtype=np.int32)
    i = sorted(rnd.randint(0, m) for _ in range(k))
    j = sorted(rnd.randint(0, n) for _ in range(k))
    pts = [[a, b] for a, b in zip(i, j)]
    if k >= 4 and rnd.random() < 0.5:
        pts[0] = [0, pts[0][1]] if rnd.random() < 0.5 else [pts[0][0], 0]
        pts[-1] = [m, pts[-1][1]] if rnd.random() < 0.5 else [pts[-1][0], n]
    if k >= 3 and rnd.random() < 0.5:           # a long horizontal (equal i) or vertical (equal j) run
        q = rnd.randrange(1, k)
        if rnd.random() < 0.5:
            pts[q][0] = pts[q - 1][0]
        else:
            pts[q][1] = pts[q - 1][1]
    if k >= 2 and rnd.random() < 0.3:
        pts[1] = list(pts[0])                    # a duplicate point
    out = [pts[0]]
    for p in pts[1:]:                            # keep the chain non-decreasing after the edits
        out.append([max(p[0], out[-1][0]), max(p[1], out[-1][1])])
    return np.array(out, dtype=np.int32).reshape(-1, 2)


def slot_tiles_bound(m, n, bw):
    """banded_slot_bytes' tile count (csrc/psa_long.cu)."""
    NB, S = (m + R - 1) // R, (n + W - 1) // W
    return min(NB * S, (n + 2 * bw * NB) // W + 2 * NB)


def rowblock_tiles(lo, hi, m, WW=W):
    """s_hi - s_lo + 1 of every row block of the 128-row grid (ChainBand::s_lo / s_hi)."""
    out = []
    for i0 in range(0, m, R):
        nr = min(R, m - i0)
        s_lo = (max(1, int(lo[i0 + 1])) - 1) // WW
        s_hi = max(s_lo, (max(1, int(hi[i0 + nr])) - 1) // WW)
        out.append(s_hi - s_lo + 1)
    return out


SHAPES = [(300, 300), (1000, 1000), (900, 120), (120, 900), (513, 257), (1, 1000), (1000, 1), (1, 1), (129, 700), (2048, 3000)]


@pytest.mark.parametrize("m,n", SHAPES)
def test_empty_chain_is_the_diagonal_band(m, n):
    for band in (0, 1, 7, 128, 300, m + n + 5):
        lo, hi = go.guide_rows(m, n, [], band)
        dlo, dhi = go.diag_rows(m, n, band)
        assert np.array_equal(lo, dlo) and np.array_equal(hi, dhi), band
        assert [tuple(x) for x in zip(lo.tolist(), hi.tolist())] == bx.band_rows(m, n, band)


@pytest.mark.parametrize("mode", [po.GLOBAL, po.LOCAL])
def test_row_oracles_equal_banded_oracles_on_the_diagonal(mode):
    rnd = random.Random(8100 + mode)
    for k in range(12):
        a, b = py_random_pair(rnd, 40, 160)
        if k % 2:
            a, b = b, a
        for band in (0, 1, 5, 17, 64, 300):
            lo, hi = go.guide_rows(len(a), len(b), [], band)
            assert go.align_rows(a, b, lo, hi, 1, 2, mode) == bo.align_banded(a, b, band, 1, 2, mode), (k, band)
            got, want = go.score_rows(a, b, lo, hi, 1, 2, mode), bo.score_banded(a, b, band, 1, 2, mode)
            assert tuple(getattr(got, f) for f in RECORD) == tuple(getattr(want, f) for f in RECORD), (k, band)


def test_random_chains_give_monotone_rows_within_the_slot_bound():
    rnd = random.Random(8200)
    for t in range(400):
        m, n = rnd.randint(1, 3000), rnd.randint(1, 3000)
        chain = random_chain(rnd, m, n, rnd.choice([1, 2, 3, 5, 16, 60]))
        bw = rnd.choice([0, 1, 7, 64, 300, 2000])
        lo, hi = go.guide_rows(m, n, chain, bw)
        assert (np.diff(lo) >= 0).all() and (np.diff(hi) >= 0).all(), (t, chain)
        assert (lo <= hi).all() and lo[0] == 0 and hi[m] == n
        assert sum(rowblock_tiles(lo, hi, m)) <= slot_tiles_bound(m, n, bw), (t, m, n, bw)
        if bw >= max(m, n):
            assert (lo == 0).all() and (hi == n).all()


def test_horizontal_run_carries_any_jump():
    # a 2000-column insertion in B at row 500 of a 1000 x 3000 pair: one row widens to cover it, band 0 still connects
    lo, hi = go.guide_rows(1000, 3000, [[500, 500], [500, 2500]], 0)
    assert (lo[500], hi[500]) == (500, 2500)
    assert (lo[499], hi[499]) == (499, 499) and (lo[501], hi[501]) == (2501, 2501)


@pytest.mark.parametrize("mode", [po.GLOBAL, po.LOCAL])
def test_exact_reference_equals_row_oracle_on_chains(mode):
    rnd = random.Random(8300 + mode)
    for k in range(40):
        a, b = py_random_pair(rnd, 30, 120)
        m, n = len(a), len(b)
        chain = random_chain(rnd, m, n, rnd.choice([0, 1, 3, 6]))
        for band in (0, 2, 9):
            lo, hi = go.guide_rows(m, n, chain, band)
            want = go.align_rows(a, b, lo, hi, 1, 2, mode)
            assert gx.align_rows(a, b, list(zip(lo.tolist(), hi.tolist())), 1, 2, mode) == want, (k, band)
            lin = go.score_rows(a, b, lo, hi, 1, 2, mode)
            assert tuple(getattr(lin, f) for f in RECORD) == tuple(getattr(want, f) for f in RECORD), (k, band)


def kernel_corner_rows(a, b, rows, g, h):
    """test_banded_range_cpu.kernel_corner over per-row bands: the global record as the kernels' int32 cells compute it."""
    m, n = len(a), len(b)
    go = g + h
    pH = [0] + [w32(-h - g * j) for j in range(1, rows[0][1] + 1)]
    pF = [KNEG] * len(pH)
    plo = 0
    for i in range(1, m + 1):
        lo, hi = rows[i]
        H, E, F = [], [], []
        for j in range(lo, hi + 1):
            if j == 0:
                H.append(w32(-h - g * i)), E.append(KNEG), F.append(KNEG)
                continue
            up = (pH[j - plo], pF[j - plo]) if 0 <= j - plo < len(pH) else (KNEG, KNEG)
            diag = pH[j - 1 - plo] if 0 <= j - 1 - plo < len(pH) else KNEG
            hl, el = (H[-1], E[-1]) if j > lo else (KNEG, KNEG)
            t1 = w32(diag + (a[i - 1] == b[j - 1]))
            e = max(w32(hl - go), w32(el - g))
            f = max(w32(up[0] - go), w32(up[1] - g))
            H.append(max(t1, e, f)), E.append(e), F.append(f)
        pH, pF, plo = H, F, lo
    c1, c2, c3 = t1, e, f
    ov = lambda v: po.NEG if v < CUT else v
    state = 1 if (c1 >= c2 and c1 >= c3) else (2 if (c2 >= c1 and c2 >= c3) else 3)
    return ov(c1), ov(c2), ov(c3), ov(max(c1, c2, c3)), state


def staircase(m, n, rnd):
    """A chain whose rows are runs that meet end to end: row i covers [c_i, c_{i+1}] (c_0 = 0, c_m = n), so a band-0
    path opens a gap on every row."""
    cuts = sorted(rnd.randint(0, n) for _ in range(m - 1))
    c = [0] + cuts + [n]
    pts = []
    for i in range(m):
        pts += [[i, c[i]], [i, c[i + 1]]]
    return np.array(pts, dtype=np.int32)


@pytest.mark.parametrize("m,n,related", [(200, 600, False), (300, 900, True), (250, 260, True)])
def test_kernel_arithmetic_exact_at_the_banded_limit_on_staircases(m, n, related):
    rnd = random.Random(8400 + m)
    rng = np.random.default_rng(m + n)
    a = random_dna(rng, m)
    b = mutated_copy(rng, a, n) if related else random_dna(rng, n)
    chain = staircase(m, n, rnd)
    for band in (0, 1):
        lo, hi = go.guide_rows(m, n, chain, band)
        rows = list(zip(lo.tolist(), hi.tolist()))
        for (g, h), over in edge_penalties(m, n):
            assert bx.span_banded(g, h, m, n) < bx.SPAN_LIMIT <= bx.span_banded(*over, m, n)
            want = gx.align_rows(a, b, rows, g, h)
            assert want.score != po.NEG
            assert kernel_corner_rows(a, b, rows, g, h) == exact_record(want), (band, g, h)


INVALID = [
    ("i above m", [[301, 5]]),
    ("j above n", [[5, 401]]),
    ("negative i", [[-1, 0]]),
    ("negative j", [[3, -2]]),
    ("i decreases", [[10, 10], [9, 20]]),
    ("j decreases", [[10, 10], [20, 9]]),
    ("late decrease", [[0, 0], [100, 100], [100, 150], [200, 140]]),
]


@pytest.mark.parametrize("name,chain", INVALID, ids=[x[0] for x in INVALID])
def test_guide_rows_rejects_invalid_chains(name, chain):
    with pytest.raises(ValueError):
        go.guide_rows(300, 400, chain, 10)


def test_guide_rows_accepts_the_edges():
    for chain in ([[0, 0]], [[300, 400]], [[0, 400]], [[300, 0], [300, 0]], [[0, 0], [0, 400], [300, 400]],
                  [[0, 0], [300, 0], [300, 400]], [[150, 200]] * 5):
        lo, hi = go.guide_rows(300, 400, chain, 3)
        assert (np.diff(lo) >= 0).all() and (np.diff(hi) >= 0).all()
