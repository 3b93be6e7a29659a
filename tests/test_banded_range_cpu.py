"""The exact banded reference (tests/banded_exact.py) against the int32 banded oracle, and the range rule of the banded
global entries against an int32 emulation of the kernels' banded cell recurrence.  No GPU.

Inside a band the full matrix's argument for check_scoring (a finite value needs at most three gap openings) does not
hold: n = 3m at band 1 needs a gap opening on every row.  The emulation below computes what sweep<> computes (int32
lanes that wrap, PSA_KNEG for the border beyond the band and for every out-of-band cell, out_value on the corner).  At
penalties the old rule admitted it reports "no path" for pairs that have one; at the largest penalties
check_banded_scoring admits it equals the exact reference."""
import random

import numpy as np
import pytest

from oracle import pyoracle as po
from tests import banded_exact as bx
from tests import banded_oracle as bo
from tests.helpers import mutated_copy, py_random_pair, random_dna
from tests.test_gpu_banded import in_band, rescore

GRID = [(1, 2), (0, 0), (0, 1), (2, 0), (3, 1), (5, 2), (1, 7), (4, 9), (0, 11)]    # test_gpu_penalties.py's WIDE
BANDS = [0, 1, 2, 5, 17, 64, 300]
RECORD = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j")

KNEG = -(1 << 29)                     # PSA_KNEG
CUT = KNEG // 4 * 3                   # out_value: below this a corner is PSA_NEG_INF

# (m, n, band, related): shapes whose band forces gap openings row after row, and mutated / square pairs
EDGE_SHAPES = [(300, 900, 1, False), (900, 300, 1, False), (400, 800, 1, False), (300, 1500, 2, False),
               (1000, 1040, 7, True), (1100, 1000, 31, True), (600, 600, 0, True)]

# the pairs the old rule admitted: (m, n, band, g, h)
OLD_RULE_CASES = [(2000, 4000, 1, 1, 500_000), (600, 1200, 1, 0, (1 << 27) - 1000), (300, 2400, 40, 0, (1 << 27) - 1400)]


def edge_pair(m, n, related, seed):
    rng = np.random.default_rng(seed)
    a = random_dna(rng, m)
    return a, (mutated_copy(rng, a, n) if related else random_dna(rng, n))


def edge_penalties(m, n):
    """The largest (g, h) check_banded_scoring admits, each with the one-unit-larger (g, h) it refuses: largest h at
    g = 0 and 3, largest g at h = 0 and 2."""
    out = []
    for g in (0, 3):
        h = bx.largest_h(m, n, g)
        out.append(((g, h), (g, h + 1)))
    for h in (0, 2):
        g = bx.largest_g(m, n, h)
        out.append(((g, h), (g + 1, h)))
    return out


def w32(x):
    return (x + (1 << 31)) % (1 << 32) - (1 << 31)


def kernel_corner(a, b, band, g, h):
    """Global record fields (t1, t2, t3, score, end_state) of the banded fill as sweep<> computes them: per cell
    t1 = diag + match, e = max(H_left - go, E_left - g), f = max(H_up - go, F_up - g), H = max(t1, e, f) in wrapping
    int32; out-of-band cells H = E = F = PSA_KNEG; borders as border_row0_H / border_col0_H inside the band; then
    global_item (out_value, end_state on the raw values)."""
    m, n = len(a), len(b)
    go = g + h
    rows = bx.band_rows(m, n, band)
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
    c1, c2, c3 = t1, e, f                   # cell (m, n) is the last cell of the last row
    ov = lambda v: po.NEG if v < CUT else v
    state = 1 if (c1 >= c2 and c1 >= c3) else (2 if (c2 >= c1 and c2 >= c3) else 3)
    return ov(c1), ov(c2), ov(c3), ov(max(c1, c2, c3)), state


def exact_record(w):
    return w.t1, w.t2, w.t3, w.score, w.end_state


@pytest.mark.parametrize("mode", [po.GLOBAL, po.LOCAL])
@pytest.mark.parametrize("g,h", GRID)
def test_exact_reference_equals_int32_oracle(mode, g, h):
    """Where int32 is exact the two restatements agree on every field: random, related (both orientations), tie-prone
    and empty pairs, bands 0 - 300."""
    rnd = random.Random(7100 + 10 * g + h + 1000 * mode)
    pairs = []
    for k in range(16):
        a, b = py_random_pair(rnd, 70, 90)
        pairs.append((a, b) if k % 2 else (b, a))
    for _ in range(4):
        m, n = rnd.randint(20, 80), rnd.randint(20, 80)
        pairs.append((bytes(rnd.choice(b"AB") for _ in range(m)), bytes(rnd.choice(b"AB") for _ in range(n))))
    pairs += [(b"AC" * 30, b"AC" * 27 + b"T"), (b"ACG" * 20, b"ACG" * 25), (b"", b"ACG"), (b"ACG", b""), (b"", b"")]
    for a, b in pairs:
        for band in BANDS:
            want = bo.align_banded(a, b, band, g, h, mode)
            got = bx.align_banded(a, b, band, g, h, mode)
            assert got == want, (a, b, band)
            lin = bo.score_banded(a, b, band, g, h, mode)
            assert tuple(getattr(got, f) for f in RECORD) == tuple(getattr(lin, f) for f in RECORD), (a, b, band)


def test_exact_reference_is_exact_past_int32():
    """A band that forces an opening on every row takes the exact score far below -2^31, where the int32 oracle
    saturates to -infinity; the exact path still re-scores to it."""
    a, b = edge_pair(600, 1200, False, 11)
    h = (1 << 27) - 1000
    w = bx.align_banded(a, b, 1, 0, h)
    assert w.score < -(1 << 31) and len(w.ops) >= 1200
    assert rescore(a, b, w.ops, w.start_i, w.start_j, 0, h, po.GLOBAL) == w.score
    assert in_band(a, b, w.ops, w.start_i, w.start_j, 1)
    assert bo.align_banded(a, b, 1, 0, h).score == po.NEG


@pytest.mark.parametrize("case", OLD_RULE_CASES, ids=["2000x4000_band1", "600x1200_band1", "300x2400_band40"])
def test_old_rule_admits_wrong_kernel_records(case):
    """The three-openings rule admits these calls; the kernels' arithmetic gets them wrong; the banded rule refuses
    them.  2000 x 4000: the exact score fits in int32 (the int32 oracle has it) but lies below out_value's cut, so the
    kernel reports no path.  The other two: the exact score is not an int32."""
    m, n, band, g, h = case
    a, b = edge_pair(m, n, False, m + band)
    assert bx.span(g, h, m, n) < bx.SPAN_LIMIT <= bx.span_banded(g, h, m, n)
    want = bx.align_banded(a, b, band, g, h)
    got = kernel_corner(a, b, band, g, h)
    assert want.score != po.NEG and got != exact_record(want)
    assert got[3] == po.NEG
    if m == 2000:
        assert po.NEG < want.score < CUT and bo.align_banded(a, b, band, g, h).score == want.score
    else:
        assert want.score < -(1 << 31)


@pytest.mark.parametrize("shape", EDGE_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}_band{s[2]}")
def test_kernel_arithmetic_exact_at_the_banded_limit(shape):
    """At the largest (g, h) the banded rule admits, the emulated kernel corner equals the exact one; with n = 3m or
    m = 3n at band 1 the exact corners reach below -2^27, so the edge is reached."""
    m, n, band, related = shape
    a, b = edge_pair(m, n, related, m + band)
    lowest = 0
    for (g, h), over in edge_penalties(m, n):
        assert bx.span_banded(g, h, m, n) < bx.SPAN_LIMIT <= bx.span_banded(*over, m, n)
        want = bx.align_banded(a, b, band, g, h)
        assert kernel_corner(a, b, band, g, h) == exact_record(want), (g, h)
        lowest = min([lowest] + [v for v in exact_record(want)[:3] if v != po.NEG])
    if band == 1 and 3 * min(m, n) == max(m, n):
        assert lowest < -(1 << 27)
        assert lowest > -(1 << 28)
